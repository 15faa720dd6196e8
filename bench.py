#!/usr/bin/env python3
"""bench.py -- env-steps/sec of the fused step kernel (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W        (N>1: launched under torch.distributed.run)
  python bench.py --impl reference ...                 (CPU arm: the fp64 oracle port on the host cores)
  python bench.py ... --dump-outputs DIR               (also write the last timed step's outputs as DIR/<name>.npy)

A "step" is one RexGymEnv.step for every environment of the batch (one kernel launch); the workload is
BASELINE.json configs[1]: 4096 envs/GPU, walk-ik, flat terrain, fused ABA+IK+motor kernel, synthetic
uniform random actions, training wrappers (ClipAction/RangeNormalize/LimitDuration) and auto-reset fused.
`value` = device-timed (CUDA events, inputs resident in HBM); `e2e` = through BatchedRexEnv.step with host
(pinned) action buffers in and obs/reward/done back out every step.  Envs shard across GPUs with no data
path collective (weak scaling).

How the K = --steps steps are timed (exactly K steps per workload; pick K large enough for the window you want):
  * the K steps are split into BLOCKS of at most 200 consecutive steps; every step is bracketed by its own pair of CUDA events
    on the launching stream with the L2 flush (256 MiB memset) between steps outside the events; a block's time is the sum of
    its event intervals;
  * before a block the stream is parked behind a device-side gate (a spin kernel a few ms long) so the host enqueues the
    whole block ahead of the GPU: no host hiccup can land between an event and its kernel;
  * per block the MAX over ranks is taken (barrier + synchronize on both sides of every block); `ms_per_step` = the sum over
    blocks / K, `value` = envs / ms_per_step.  The mean over the whole window, not a median over blocks: the step's cost
    follows the gait phase of the batch, so blocks at different points of the window differ systematically, not by noise.
    `timing` lists every block and every rank's own time per step;
  * the clocks come from ONE `nvidia-smi -lms 200` process per rank started before and stopped after the timed region
    (the profiling recipe's form), not from a process spawned every 200 ms.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
WORKLOAD = dict(task="walk", signal_type="ik", terrain_type="plane", target_position=2.0, backwards=False,
                normalize=True, max_episode_steps=2000, auto_reset=True)
# wall seconds per simulated second of the reference's own README recording (tests/test_readme_gif_clock.py: >= 3.6)
DEMO_CLOCK = 4.0
BLOCK_STEPS = 200


def b_alg(num_motors, A, O):
    """Algorithmic bytes per env-step (SURVEY.md section 8(d), for the state layout actually built): state words read once
    and written once (43 float + 14 int; the arm adds 12 float + 2 int), + actions, obs, reward, done, last command."""
    words = (43 + 14) if num_motors == 12 else (55 + 16)
    return 2 * words * 4 + A * 4 + O * 4 + 4 + 1 + num_motors * 4


class ClockSampler(object):
    """One `nvidia-smi -lms 200` child for this rank's GPU, alive only around the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_id):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_id), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        try:
            self.p.terminate()
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            try:
                self.p.kill()
            except Exception:
                pass
            out = ""
        rows = [[x.strip() for x in l.split(",")] for l in out.strip().splitlines()]
        rows = [r for r in rows if len(r) >= 6 and r[0].isdigit()]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(r[2 + k].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(int(r[1]) for r in rows if r[1].isdigit()), "reasons": reasons,
                "samples": len(rows)}


def split_blocks(K):
    """Sizes of the blocks K timed steps are split into: as even as possible, at most BLOCK_STEPS each, summing to K."""
    nb = -(-K // BLOCK_STEPS)
    return [K // nb + (1 if b < K % nb else 0) for b in range(nb)]


def stagger_episodes(env, acts, span=256, groups=32):
    """Untimed: spread the episode ages of the batch uniformly over `span` control steps (reset 1/groups of the envs, step
    span/groups times, repeat).  After a common reset every env is in the same phase of the gait ramp and the step kernel's
    cost follows that phase; an auto-resetting training batch is de-synchronised, so the timed window should be too --
    whatever --steps the caller picks."""
    import torch
    n = env.num_envs
    perm = torch.randperm(n, device=env.device, generator=torch.Generator(device=env.device).manual_seed(7))
    per = (n + groups - 1) // groups
    k = 0
    for g in range(groups):
        idx = perm[g * per:(g + 1) * per].to(torch.int32)
        if idx.numel():
            env.reset(idx)
        for _ in range(span // groups):
            env.step(acts[k % acts.shape[0]]); k += 1


class Timer(object):
    """Device-timed blocks of consecutive steps (see the module docstring).  `last` holds what env.step returned in the
    most recent timed step."""

    def __init__(self, dev, world, flush):
        import torch
        self.torch, self.dev, self.world, self.flush = torch, dev, world, flush
        self.clock_hz = 1.9e9
        self.last = None

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def block(self, env, acts, first, K, after_step=None, done_acc=None):
        torch = self.torch
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        self.barrier()
        torch.cuda._sleep(int(self.clock_hz * (2e-3 + K * 6e-5)))       # the gate: the host enqueues the block ahead of the GPU
        for k in range(K):
            self.flush.zero_()                                          # L2 flush between timed iterations (not timed)
            ev[k][0].record()
            self.last = env.step(acts[(first + k) % acts.shape[0]])
            if after_step is not None:
                after_step(env)
            ev[k][1].record()
            if done_acc is not None:
                done_acc.add_(self.last[2].sum())
        self.barrier()
        return sum(a.elapsed_time(b) for a, b in ev)

    def run(self, env, acts, first, K, after_step=None):
        """Exactly K timed steps -> dict(ms_per_step, block_ms [max over ranks per block], per_rank_ms_per_step,
        resets_per_step, launches)."""
        torch = self.torch
        done_acc = torch.zeros((), dtype=torch.int64, device=self.dev)
        l0 = env.launch_count
        sizes, mine = split_blocks(K), []
        for kb in sizes:
            mine.append(self.block(env, acts, first + sum(sizes[:len(mine)]), kb, after_step, done_acc))
        launches = env.launch_count - l0
        mine_t = torch.tensor(mine, dtype=torch.float64, device=self.dev)
        per_block = mine_t.clone()
        per_rank = [float(mine_t.sum()) / K]
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(per_block, op=dist.ReduceOp.MAX)
            g = [torch.zeros_like(mine_t) for _ in range(self.world)]
            dist.all_gather(g, mine_t)
            per_rank = [float(x.sum()) / K for x in g]
        dn = done_acc.to(torch.float64)
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(dn)
        return {"ms_per_step": float(per_block.sum()) / K, "block_ms": [round(float(x), 5) for x in per_block], "block_steps": sizes, "blocks": len(sizes),
                "window_ms": round(float(per_block.sum()), 3), "per_rank_ms_per_step": [round(x, 6) for x in per_rank],
                "resets_per_step": float(dn) / (self.world * env.num_envs * K), "launches": int(launches), "steps_timed": K}


def run_reference(args):
    """CPU arm: the reference's CPU path.  pybullet is not installable here (no network, not in the wheelhouse),
    so this times the fp64 oracle port of the same path (oracle/, kind='port') with all host threads, on a
    bounded sample of the workload (32 envs per thread per step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.oracle import OracleSim
    try:
        cores = len(os.sched_getaffinity(0))        # cores this process may actually use (cgroup/affinity aware)
    except AttributeError:
        cores = os.cpu_count() or 1
    try:                                            # a cgroup CPU quota below the affinity count would oversubscribe
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            cores = min(cores, max(1, int(int(q) / int(p))))
    except Exception:
        pass
    cores = max(1, min(cores, 64))
    os.environ.setdefault("OMP_WAIT_POLICY", "passive")
    n = 32 * cores                                  # 32 envs per thread per step keeps the fork/join overhead small
    sim = OracleSim(n, "walk", "ik", target_position=2.0, backwards=False, normalize=True, max_episode_steps=2000)
    sim.reset()
    rng = np.random.default_rng(1234)
    acts = rng.uniform(-1, 1, size=(args.steps + args.warmup, n, sim.A)).astype(np.float32)
    for k in range(args.warmup):
        _, _, d = sim.step(acts[k], nthreads=cores)
        if d.any():
            sim.reset(np.nonzero(d)[0])
    t0 = time.perf_counter()
    for k in range(args.warmup, args.warmup + args.steps):
        o, r, d = sim.step(acts[k], nthreads=cores)
        if d.any():
            sim.reset(np.nonzero(d)[0])
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"observ": o, "reward": r, "done": d})
    v = n * args.steps / dt
    cb = {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port",
          "sample": f"{n} envs x {args.steps} steps of the walk-ik flat workload, OpenMP over envs; NOT PyBullet (not installable "
                    "here): the fp64 C restatement of the same path"}
    print(json.dumps({"impl": "reference", "metric": "env-steps/sec", "value": v, "unit": "env-steps/s",
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                      "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": f"walk-ik flat, {n}-env sample per step, fp64 CPU port of the path on {cores} threads"},
                      "cpu_baseline": cb,
                      "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def cpu_baseline_leg():
    from oracle.oracle import OracleSim
    n, steps = 64, 200
    sim = OracleSim(n, "walk", "ik", target_position=2.0, backwards=False, normalize=True, max_episode_steps=2000)
    sim.reset()
    rng = np.random.default_rng(1234)
    acts = rng.uniform(-1, 1, size=(steps, n, sim.A)).astype(np.float32)
    t0 = time.perf_counter()
    for k in range(steps):
        _, _, d = sim.step(acts[k], nthreads=1)
        if d.any():
            sim.reset(np.nonzero(d)[0])
    dt = time.perf_counter() - t0
    return {"value": n * steps / dt, "unit": "env-steps/s", "cores": 1, "kind": "port",
            "sample": f"{n} envs x {steps} steps of the same walk-ik workload, single thread, fp64 oracle port (not PyBullet)"}


def kernel_counts():
    """Per-env-step instruction / flop counts of the step kernel from this round's ncu capture (profiles/kernel_counts.json,
    written by tools/ncu_summary.py): the numerators of the issue-rate and fp32 roofline fractions."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "kernel_counts.json")))
    except Exception:
        return {}


def dump_outputs(out_dir, arrays, rank=None):
    """Write the last timed step's outputs as float32 DIR/<name>.npy (DIR/<name>_rank<r>.npy when sharded over ranks)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ("" if rank is None else "_rank%d" % rank) + ".npy"), np.asarray(a, np.float32))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--envs-per-gpu", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-extras", action="store_true", help="headline + e2e only (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after timing, write what the last timed step returned (observ, reward, done, motor command) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL prints its version banner on stdout when the communicator comes up: keep stdout for the ONE JSON line
        sys.stdout.flush()
        saved = os.dup(1); os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize(dev)
        finally:
            sys.stdout.flush(); os.dup2(saved, 1); os.close(saved)
    import rex_gym_b200 as R
    from rex_gym_b200 import sharding
    n = args.envs_per_gpu
    W = max(args.warmup, 3)
    K = args.steps
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)        # > 126 MB L2
    T = Timer(dev, world, flush)
    gen = torch.Generator(device=dev); gen.manual_seed(1234 + rank)
    try:
        gpu_id = "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
    except Exception:
        gpu_id = str(local)

    def measure(kw, nb, Kb, after_step=None, n_act=None):
        """Create, de-synchronise, warm up and time one workload; returns the Timer dict + error flags."""
        env = R.BatchedRexEnv(num_envs=nb, device=f"cuda:{local}", seed=1234, env_offset=rank * nb, **kw)
        env.reset()
        acts = torch.rand((n_act or 32, nb, env.action_dim), device=dev, generator=gen) * 2 - 1      # resident in HBM
        stagger_episodes(env, acts)
        for k in range(W):
            env.step(acts[k % acts.shape[0]])
        r = T.run(env, acts, W, Kb, after_step=after_step)
        r["error_flags_or"] = env.check_errors()
        r["envs_per_gpu"], r["value"], r["unit"] = nb, world * nb * 1e3 / r["ms_per_step"], "env-steps/s"
        return env, acts, r

    # ---- device-timed headline --------------------------------------------------------------------------------------
    sampler = ClockSampler(gpu_id)
    env, acts, head = measure(WORKLOAD, n, K, n_act=max(32, min(W + K, 256)))
    A, O = env.action_dim, env.obs_dim
    value, ms_per_step = head["value"], head["ms_per_step"]
    if args.dump_outputs:                   # what BatchedRexEnv.step handed its caller; info[i]["action"] = motor command row i
        obs, reward, done, _ = T.last
        dump_outputs(args.dump_outputs, {"observ": obs.cpu().numpy(), "reward": reward.cpu().numpy(), "done": done.cpu().numpy(),
                                         "motor_command": env.last_command().t().cpu().numpy()}, rank if world > 1 else None)

    # ---- end-to-end arm: host buffers through the public API, copies inside the timed region (the same K steps in the
    # same blocks, wall clock) ----
    acts_h = acts.cpu().numpy()
    for k in range(3):
        env.step(acts_h[k])
    e2e_blocks, k = [], 0
    for kb in split_blocks(K):
        T.barrier()
        t0 = time.perf_counter()
        for _ in range(kb):
            o, r, d, _ = env.step(acts_h[(W + k) % acts_h.shape[0]])
            k += 1
        T.barrier()
        tl = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        e2e_blocks.append(float(tl.item()))
    e2e_value = world * n * K / sum(e2e_blocks)
    clocks = sampler.stop()
    err = env.check_errors()
    env.close()

    extras = {}
    if not args.no_extras:
        def extra(name, kw, nb, after_step=None, note=None):
            try:
                e, _, r = measure(kw, nb, K, after_step=after_step)
                e.close()
                keep = {k: r[k] for k in ("envs_per_gpu", "ms_per_step", "value", "unit", "resets_per_step", "error_flags_or", "blocks", "window_ms")}
                keep["global_envs"], keep["steps"] = world * nb, K
                if note:
                    keep["note"] = note
                extras[name] = keep
            except Exception as ex:                                    # an extra must never take the headline down with it
                extras[name] = {"error": repr(ex)}
        common = dict(normalize=True, max_episode_steps=2000, auto_reset=True)
        # the same walk-ik workload at the clock of the reference's own README recording (robots walk to the goal instead of
        # tipping over at step ~240), and the north-star size at the three clocks
        extra("walk_ik_demo_clock_x4", dict(WORKLOAD, gait_clock_scale=DEMO_CLOCK), n)
        extra("north_star_size", WORKLOAD, 65536)
        extra("north_star_size_demo_clock_x4", dict(WORKLOAD, gait_clock_scale=DEMO_CLOCK), 65536)
        extra("north_star_size_training_clock_x9", dict(WORKLOAD, gait_clock_scale=9.0), 65536)     # walk-ik training runs: DESIGN.md section 2
        # BASELINE.json configs[2..4]
        extra("C3_gallop_ol_rand_gains", dict(common, task="gallop", signal_type="ol", motor_kp_range=(0.8, 1.2), motor_kd_range=(0.01, 0.03)), 16384)
        c4 = 65536 // world if world >= 4 else 16384
        extra("C4_turn_ik_heightfield", dict(common, task="turn", signal_type="ik", terrain_type="random", num_fields=64), c4,
              note="BASELINE configs[3]: 65536 envs sharded over 4 GPUs" + ("" if world == 4 else f" (here {world} GPU(s) x {c4})"))
        c5 = 131072 // world if world == 8 else 16384
        ag = None
        if world > 1:
            def ag(e):                                                 # the one collective of the path, INSIDE the timed step
                sharding.all_gather_outputs(e._obs, e._reward, e._done_u8)
        extra("C5_standup_arm_18dof", dict(common, task="standup", signal_type="ol", mark="arm"), c5, after_step=ag,
              note="BASELINE configs[4]: 131072 envs on 8 GPUs, NCCL all-gather of the packed outputs inside every timed step"
                   + ("" if world == 8 else f" (here {world} GPU(s) x {c5}" + (", no collective at 1 GPU)" if world == 1 else ")")))
        # SURVEY 8(f) rows 1-2: the all-device rollout (policy inference + env step + filter update per control step,
        # one CUDA graph per 32-step window), same workload
        def rollout_extra(name, nr, tensor_cores):
            try:
                from rex_gym_b200.agents import ForwardGaussianPolicy, Rollout
                envr = R.BatchedRexEnv(num_envs=nr, device=f"cuda:{local}", seed=1234, env_offset=rank * nr, **WORKLOAD)
                net = ForwardGaussianPolicy(envr.obs_dim, envr.action_dim, device=f"cuda:{local}", tensor_cores=tensor_cores)
                ro = Rollout(envr, net, 32, seed=1234, training=True, use_graph=True)
                perm = torch.randperm(nr, device=dev, generator=torch.Generator(device=dev).manual_seed(7))
                for g in range(8):                  # de-synchronise the episodes: 8 groups, 32 control steps apart (untimed)
                    idx = perm[g * nr // 8:(g + 1) * nr // 8]
                    ro._cur[idx] = envr.reset(idx.to(torch.int32))
                    ro.collect()
                T.barrier()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(20):
                    ro.collect()
                b.record(); T.barrier()
                tr = torch.tensor([a.elapsed_time(b)], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(tr, op=dist.ReduceOp.MAX)
                extras[name] = {
                    "what": "ForwardGaussianPolicy(200-100) perform + env step + filter update per control step, CUDA graph of 32 steps"
                            + ("; policy / value layer 2 on the tensor cores (tcgen05 kind::tf32)" if tensor_cores else "; networks in fp32 on the CUDA cores"),
                    "envs_per_gpu": nr, "ms_per_control_step": float(tr.item()) / 640,
                    "value": world * nr * 640 / (float(tr.item()) * 1e-3), "unit": "env-steps/s", "kernels_per_control_step": 3}
                envr.close(); net.close()
            except Exception as e:
                extras[name] = {"error": repr(e)}
        rollout_extra("rollout_with_policy", n, False)
        rollout_extra("rollout_with_policy_65536", 65536, False)
        rollout_extra("rollout_with_policy_65536_tf32_tensor_cores", 65536, True)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        sm_mhz = float(clocks.get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0)
        per_launch_s = ms_per_step * 1e-3
        achieved = n * b_alg(12, A, O) / per_launch_s / 1e9
        kc = kernel_counts().get("walk_ik_plane", {})
        roof = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of one step_kernel launch at 4096 envs from this round's
                # `ncu --set full` capture (profiles/kernel_counts.json names the file); the 1 MB state stays in the 126 MB L2
                "traffic": kc.get("dram_bytes_per_launch_4096") if n == 4096 else None, "of": "measured" if peaks else "fallback",
                "note": "mandated HBM roofline; the state fits L2 and the kernel is issue / dependent-latency bound -- see `issue` and `fp32`"}
        if kc.get("warp_inst_per_env_step"):
            ipeak = 148 * 4 * sm_mhz * 1e6                              # 4 schedulers per SM, one warp instruction per clock each
            ia = value / world * kc["warp_inst_per_env_step"]
            roof["issue"] = {"achieved": ia, "peak": ipeak, "unit": "warp-inst/s", "frac": ia / ipeak,
                             "per_env_step": kc["warp_inst_per_env_step"], "source": kc.get("source")}
        if kc.get("flop_per_env_step"):
            fpeak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12                  # 128 fp32 lanes per SM, FMA = 2 flop
            fa = value / world * kc["flop_per_env_step"] / 1e12
            roof["fp32"] = {"achieved": fa, "peak": fpeak, "unit": "TFLOP/s", "frac": fa / fpeak,
                            "per_env_step": kc["flop_per_env_step"], "source": kc.get("source")}
        line = {
            "metric": "env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{n} envs/GPU walk-ik flat terrain, fused ABA+IK+motor kernel (BASELINE configs[1]), gait clock = simulation clock",
                       "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"env-sharded x{world}, no data-path collective",
                       "wrappers": "ClipAction+RangeNormalize+LimitDuration(2000)+auto-reset fused", "l2": "flushed between timed steps (256 MiB memset)",
                       "episode_phase": "ages staggered uniformly over 256 control steps before the warm-up (de-synchronised batch, as under auto-reset)",
                       "resets_per_step": head["resets_per_step"],
                       "resets_note": "fraction of env-steps that ended an episode (in-kernel auto-reset: a snapshot copy, cost included). At the "
                                      "simulation clock this model's forward trot tips over after ~240 control steps (1/240 = 0.0042); at the clock "
                                      "the reference's README recording ran at (x4, extras) it walks to the goal",
                       "error_flags_or": err, "extras": extras},
            "timing": {"steps_timed": head["steps_timed"], "block_steps": head["block_steps"], "blocks": head["blocks"],
                       "window_ms": head["window_ms"], "block_ms": head["block_ms"], "per_rank_ms_per_step": head["per_rank_ms_per_step"],
                       "statistic": "sum over blocks of the max over ranks, / steps_timed",
                       "e2e_blocks": len(e2e_blocks), "e2e_window_ms": round(1e3 * sum(e2e_blocks), 3)},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": n * A * 4,
                    "d2h_bytes_per_step": n * (O * 4 + 4 + 1) + 4},
            "gpu_launches": head["launches"],
            "roofline": roof,
        }
        try:
            line["cpu_baseline"] = cpu_baseline_leg()
        except Exception as e:  # the checker library is test infrastructure; report rather than die
            line["cpu_baseline"] = {"value": None, "unit": "env-steps/s", "cores": 1, "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
