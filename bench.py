#!/usr/bin/env python
"""bench.py — env-steps/s of the A1 hot path (BASELINE.json configs[1]: 4096 parallel A1 envs, flat terrain, fixed
ETG + random residual policy rollout) on N B200s of one node, with the roofline of the dominant kernel and the CPU
oracle timed beside it.

  python bench.py [--gpus N] [--steps K] [--warmup W]              # torchrun launches one rank per GPU for N>1
  python bench.py --impl reference [--gpus N] [--steps K] ...      # the CPU arm (oracle port; pybullet is absent)
  python bench.py ... --dump-outputs DIR                           # also save what the last timed step returned, DIR/<name>.npy

A "step" is one env.step() over the whole env batch of a rank (= 13 fused physics substeps + ETG + obs/reward pack in
ONE kernel launch).  Weak scaling: every rank owns its own 4096 envs, no data-path collective.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
WORKLOAD = "BASELINE configs[1]: 4096 parallel A1 envs per GPU, flat terrain, fixed ETG (Opt_with_points 0.1/0.05) + uniform(-0.3,0.3) residual rollout, auto-reset on fall"
# algorithmic HBM bytes per env-step of b2q_step_kernel<float> (DESIGN.md §5): every per-env array touched once
ALG_BYTES_IN = 21 * 16 + 15 * 16 + 16 * 16 + 48 + 4 + 2 * 3 * 4 * 16      # state, params, ETG, action, counter, history reads
ALG_BYTES_OUT = 21 * 16 + 2 * 3 * 4 * 16 + 49 * 4 + 4 + 1 + 56 * 4 + 4      # state, history writes, obs, reward, done, info, counter
ALG_BYTES_PER_ENV_STEP = ALG_BYTES_IN + ALG_BYTES_OUT
DUMP_BYTES = 60 * 10 ** 6                    # --dump-outputs payload cap: the files, headers included, stay under 64 MB


def etg_weights():
    from paddlerobotics_b200.etg import ETG_layer, Opt_with_points
    layer = ETG_layer(0.5, 0.026, 20, 0.04, np.array([-np.pi / 2, 0]), 0.2, 0.5)
    w, b, _ = Opt_with_points(ETG=layer, ETG_T=0.5, Footheight=0.1, Steplength=0.05)   # train.py:298-299 (BASELINE.md §3.3)
    return w, b


class ClockSampler(threading.Thread):
    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu, self.rows, self._halt = gpu, [], threading.Event()

    def run(self):
        # NVML directly (5 ms period: the timed region is only ~0.1 s long); nvidia-smi subprocess as the fallback
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            bits = ((0x8, 2), (0x40, 3), (0x20, 4), (0x4, 5))     # hw_slowdown, hw_thermal_slowdown, sw_thermal_slowdown, sw_power_cap
            while not self._halt.is_set():
                r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)), str(mx), "", "", "", ""]
                for bit, col in bits:
                    row[col] = "Active" if (r & bit) else "Not Active"
                self.rows.append(row)
                self._halt.wait(0.005)
            return
        except Exception:
            pass
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def host_threads():
    """Usable host threads: the scheduler affinity, capped by the cgroup CPU quota when one is set."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def cpu_oracle_rate(n_envs, steps, threads, w, b, seed=1234):
    """Oracle (float64 C port of the path; pybullet/rlschool are absent) on `threads` host threads: every thread owns a
    contiguous slice of envs and runs `steps` control steps on it (one env per actor, as Dynamic_parallel_model.py:96-99)."""
    from oracle import oracle as O
    batch = O.OracleBatch(n_envs, etg_w=w, etg_b=b)
    rng = np.random.default_rng(seed)
    batch.rollout(rng.uniform(-0.3, 0.3, (2, n_envs, 12)), auto_reset=True, nthreads=threads)      # warm
    acts = rng.uniform(-0.3, 0.3, (steps, n_envs, 12))
    t0 = time.perf_counter()
    batch.rollout(acts, auto_reset=True, nthreads=threads)
    dt = time.perf_counter() - t0
    return n_envs * steps / dt, dt


def dump_outputs(out_dir, outputs, suffix=""):
    """Saves the arrays one env.step() returned as out_dir/<name><suffix>.npy in float32, so that two builds can be compared output for
    output.  Above DUMP_BYTES in all, a fixed seeded sample of env rows (the same rows for the same env count) stands for the batch."""
    n = next(iter(outputs.values())).shape[0]
    row_bytes = 4 * sum(t[0].numel() for t in outputs.values())
    keep = min(n, DUMP_BYTES // row_bytes)
    rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if keep < n else slice(None)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), t.float().cpu().numpy()[rows])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    w, b = etg_weights()
    rate1, _ = cpu_oracle_rate(64, 6, 1, w, b)
    W, K = max(args.warmup, 1), args.steps
    budget_s = 150.0                                          # the whole --steps/--warmup run must end within a few minutes on any host
    est = rate1 * threads * 0.7                               # env-steps/s this host should reach
    # the SAME workload as the GPU arm (one step = 4096 envs) whenever (W + K) such steps fit the budget; only a host too slow for that
    # falls back to a bounded sample of the env batch per step (throughput per env is the same: every thread stays saturated)
    n_envs = ENVS_PER_GPU if (W + K) * ENVS_PER_GPU / est <= budget_s else int(max(8 * threads, budget_s * est / (W + K)))
    from oracle import oracle as O
    batch = O.OracleBatch(n_envs, etg_w=w, etg_b=b)
    rng = np.random.default_rng(1234)
    batch.rollout(rng.uniform(-0.3, 0.3, (W, n_envs, 12)), auto_reset=True, nthreads=threads)
    acts = rng.uniform(-0.3, 0.3, (K, n_envs, 12))
    t0 = time.perf_counter()
    batch.rollout(acts, auto_reset=True, nthreads=threads)
    dt = time.perf_counter() - t0
    val = n_envs * K / dt
    line = {
        "impl": "reference", "metric": "env-steps/sec (A1, 4096 envs)", "value": val, "unit": "env-steps/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": 1e3 * dt / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": n_envs, "substeps_per_step": 13, "solver_iters": 23,
                   "note": "CPU oracle (Bullet-style float64 restatement), NOT pybullet: pybullet/rlschool are absent from the image; %s" % ("full 4096-env workload per step" if n_envs == ENVS_PER_GPU else "bounded sample of %d envs per step (host too slow for 4096 x %d steps in %.0f s)" % (n_envs, K, budget_s))},
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port", "per_thread": val / threads, "single_thread": rate1,
                         "sample": "%d envs x %d control steps, %d pthreads (one contiguous env slice per thread)" % (n_envs, K, threads)},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def _max_over_ranks(x, dev, world):
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def run_extras(args, rank, world, local, dev, w, b):
    """BASELINE configs[2..4] and the strong-scaling form of configs[1]/[4], measured in the same run on the same N ranks (VERDICT r1 #3):
    every number is device-timed (CUDA events, max over ranks) except the ES generation, which includes host work and is wall-clocked
    between synchronised barriers."""
    import torch
    import torch.distributed as dist
    from paddlerobotics_b200.agent import MujocoAgent, SACLearner
    from paddlerobotics_b200.env import VecQuadrupedalEnv
    from paddlerobotics_b200.es import PopulationEvaluator, SimpleGA, solutions_to_etg_device
    from paddlerobotics_b200.etg import ETG_layer, Opt_with_points, shipped_gait
    from paddlerobotics_b200.terrain import make_terrain
    out = {"n_ranks": world}
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)

    def rollout_rate(env, n_local, K, W=20, amp=0.3):
        g = torch.Generator(device=dev); g.manual_seed(99 + rank)
        pool = (torch.rand(32, n_local, 12, device=dev, generator=g) * 2 - 1) * amp
        for k in range(W):
            env.step(pool[k % 32])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for k in range(K):
            flush.zero_()
            ev[k][0].record(); env.step(pool[(W + k) % 32]); ev[k][1].record()
        torch.cuda.synchronize()
        ms = _max_over_ranks(sum(a.elapsed_time(c) for a, c in ev), dev, world)
        return ms / K

    # (i) strong scaling of configs[1]: 4096 envs IN TOTAL, 4096/N per rank, flat terrain
    n_local = ENVS_PER_GPU // world
    env = VecQuadrupedalEnv(n_local, device=local, auto_reset=True); env.reset(w, b)
    ms = rollout_rate(env, n_local, 200)
    out["strong_scaling_flat"] = {"envs_total": ENVS_PER_GPU, "envs_per_rank": n_local, "ms_per_step": ms, "value": ENVS_PER_GPU / (ms * 1e-3), "unit": "env-steps/s",
                                  "note": "fixed total work; the driver's speed-up is value(N)/value(1)"}
    env.close()
    # (i') the same at a batch that fills the GPU: 65536 envs in total (8192 per rank at N = 8) — where strong scaling is NOT capped by the
    # single-warp latency floor of the step kernel (DESIGN.md §5)
    n_big = 65536 // world
    env = VecQuadrupedalEnv(n_big, device=local, auto_reset=True); env.reset(w, b)
    ms = rollout_rate(env, n_big, 60, W=10)
    out["strong_scaling_flat_65536"] = {"envs_total": 65536, "envs_per_rank": n_big, "ms_per_step": ms, "value": 65536 / (ms * 1e-3), "unit": "env-steps/s"}
    env.close()
    # (iv) configs[4]: stairs height field (make_terrain('stairstair'), train.py:48-50 parameters), 4096 envs in total, strong scaling;
    # the reference's shipped walking gait drives the robots onto the stairs, starts spread over +-0.3 m (reset(x_noise))
    ws, bs = shipped_gait()
    env = VecQuadrupedalEnv(n_local, device=local, auto_reset=True, heightfield=make_terrain("stairstair"), body_collisions=1, max_episode_steps=400)
    g = torch.Generator(device=dev); g.manual_seed(5 + rank)
    env.reset(ws, bs, x_offset=torch.rand(n_local, device=dev, generator=g) * 0.6 - 0.1)
    for k in range(100):                                          # walk to the staircase before timing (2.6 s of simulated time)
        env.step(torch.zeros(n_local, 12, device=dev))
    ms = rollout_rate(env, n_local, 200, amp=0.03)               # small residuals: the shipped gait keeps walking (it falls within ~12 steps at +-0.3)
    st = env.get_state()
    out["strong_scaling_stairs"] = {"envs_total": ENVS_PER_GPU, "envs_per_rank": n_local, "ms_per_step": ms, "value": ENVS_PER_GPU / (ms * 1e-3), "unit": "env-steps/s",
                                    "terrain": "stairstair height field 0.02 m cells, step 0.08 x 0.30 m x 5 up / 5 down",
                                    "frac_envs_past_first_step": float((st[:, 0] > 0.8).float().mean()), "mean_base_height": float(st[:, 2].mean())}
    env.close()
    # (ii) configs[2]: one ES generation, pop 256 x 16 rollouts x 400 steps, individuals sharded whole over the ranks, ONE all-gather
    pop, roll, T = 256, 16, 400
    layer = ETG_layer(0.5, 0.026, 20, 0.04, np.array([-np.pi / 2, 0]), 0.2, 0.5)
    w0, b0, pts = Opt_with_points(ETG=layer, ETG_T=0.5, Footheight=0.1, Steplength=0.05)
    np.random.seed(0)                                            # identical populations on every rank (SimpleGA draws from the global RNG, es.py:259-271)
    ga = SimpleGA(12, sigma_init=0.02, sigma_decay=0.99, sigma_limit=0.005, elite_ratio=0.1, weight_decay=0.005, popsize=pop, param=np.zeros(12))
    ev = PopulationEvaluator(pop, roll, max_steps=T, rank=rank, world=world, device=local)
    gens, t_gen, t_gather = 3, [], []
    for gi in range(gens + 1):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        sol = ga.ask()
        wsd, bsd = solutions_to_etg_device(sol, pts, w0, b0, device=local)
        fit, mlen = ev.evaluate(wsd.cpu().numpy(), bsd.cpu().numpy())
        fit_h = fit.double().cpu().numpy()
        ga.tell(fit_h)
        torch.cuda.synchronize()
        dt = _max_over_ranks(time.perf_counter() - t0, dev, world)
        if gi > 0:
            t_gen.append(dt)
    if world > 1:                                                # the collective alone: [world, 2, pop/world] floats
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        buf = torch.empty(world, 2, pop // world, device=dev)
        for _ in range(5):
            dist.all_gather_into_tensor(buf, ev._fl.reshape(1, 2, -1))
        torch.cuda.synchronize(); e0.record()
        for _ in range(50):
            dist.all_gather_into_tensor(buf, ev._fl.reshape(1, 2, -1))
        e1.record(); torch.cuda.synchronize()
        t_gather = _max_over_ranks(e0.elapsed_time(e1) / 50 * 1e3, dev, world)
    chk = torch.tensor(fit_h, device=dev)
    same = True
    if world > 1:
        ref = chk.clone(); dist.broadcast(ref, 0); same = bool(torch.equal(ref, chk))
    out["es_generation"] = {"popsize": pop, "rollouts": roll, "steps": T, "envs_per_rank": pop * roll // world, "s_per_generation": float(np.mean(t_gen)),
                            "generations_per_s": 1.0 / float(np.mean(t_gen)), "env_steps_per_s": pop * roll * T / float(np.mean(t_gen)),
                            "allgather_us": t_gather if world > 1 else None, "allgather_bytes": 2 * pop * 4, "fitness_identical_on_every_rank": same,
                            "includes": "SimpleGA.ask, on-device Opt_with_points for 256 individuals, reset, 400 control steps + per-step return accumulation, fitness kernel, ONE all-gather of [fitness|length], tell"}
    ev.env.close()
    # (iii) configs[3]: SAC learn, global batch 8192 = 8192/N per rank, ONE flat gradient bucket all-reduced (NCCL) between gradient and Adam phases
    B = 8192 // world
    ag = MujocoAgent(49, 12, device=local, seed=3)
    L = SACLearner(ag, B, world=world, sync="flat")
    d = lambda *sh: torch.randn(*sh, device=dev)
    o, no, ac, r, t = d(B, 49), d(B, 49), torch.rand(B, 12, device=dev) * 2 - 1, d(B), torch.ones(B, device=dev)
    e1_, e2_ = d(B, 12), d(B, 12)
    for _ in range(5):
        L.learn(o, ac, r, no, t, eps_next=e1_, eps_cur=e2_, pull=False)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    it = 30
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(it)]
    ar = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(it)]
    for k in range(it):
        L.allreduce_events = ar[k] if world > 1 else None
        evs[k][0].record(); L.learn(o, ac, r, no, t, eps_next=e1_, eps_cur=e2_, pull=False); evs[k][1].record()
    torch.cuda.synchronize()
    learn_us = _max_over_ranks(sum(a.elapsed_time(c) for a, c in evs) / it * 1e3, dev, world)
    ar_us = _max_over_ranks(sum(a.elapsed_time(c) for a, c in ar) / it * 1e3, dev, world) if world > 1 else None
    out["sac_learn"] = {"global_batch": 8192, "batch_per_rank": B, "us_per_learn": learn_us, "allreduce_us": ar_us, "allreduce_floats": L.na + L.nc,
                        "samples_per_s": 8192 / (learn_us * 1e-6), "sync": "flat: critic + actor gradients against the pre-update parameters, ONE ncclAllReduce(avg) of [actor|critic], then both Adam steps + Polyak",
                        "launches_per_learn": None}
    l0 = int(L.lib.b2q_sac_launch_count(L.h)); L.learn(o, ac, r, no, t, eps_next=e1_, eps_cur=e2_, pull=False)
    out["sac_learn"]["launches_per_learn"] = int(L.lib.b2q_sac_launch_count(L.h)) - l0
    L.close()
    if world == 1:
        # single-GPU production path: the reference's update order (sac.py:77-118) replayed from ONE CUDA graph, batch gathered straight into
        # the graph's static inputs, rsample() noise from the counter RNG inside the kernels (no per-step torch kernels at all)
        L = SACLearner(MujocoAgent(49, 12, device=local, seed=3), B)
        for x, sx in zip((o, ac, r, no, t), L.static_batch()):
            sx.copy_(x)
        sb = L.static_batch()
        for _ in range(5):
            L.learn(*sb, graph=True, pull=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            L.learn(*sb, graph=True, pull=False)
        e1.record(); torch.cuda.synchronize()
        out["sac_learn"]["us_per_learn_cuda_graph"] = e0.elapsed_time(e1) / 50 * 1e3
        L.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=40)
    ap.add_argument("--impl", type=str, default="b2q")
    ap.add_argument("--envs", type=int, default=ENVS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the BASELINE configs[2..4] / strong-scaling block")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write obs / reward / done / info of the last timed step to DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the GPU path's outputs; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU: there is no CPU fallback for the product path"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from paddlerobotics_b200.env import VecQuadrupedalEnv
    W, K, n = max(args.warmup, 3), args.steps, args.envs
    w, b = etg_weights()
    env = VecQuadrupedalEnv(n, device=local, auto_reset=True)
    env.reset(w, b)
    dev = env.device
    # residual actions: uniform(-0.3, 0.3), counter-based per (seed, rank, step) pool resident in HBM
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    pool = torch.rand(64, n, 12, device=dev, generator=g) * 0.6 - 0.3
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev, dtype=torch.float32)     # > 126 MB L2
    for k in range(W):
        env.step(pool[k % 64])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    l0 = env.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    torch.cuda.synchronize()
    for k in range(K):
        flush.zero_()                                        # evict the env state from L2 (outside the event pair)
        ev[k][0].record()
        env.step(pool[(W + k) % 64])
        ev[k][1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches = env.launch_count() - l0
    total_ms = sum(a.elapsed_time(bb) for a, bb in ev)
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t[0])
    value = world * n * K / (total_ms * 1e-3)
    done_frac = float(env.done.float().mean())
    if args.dump_outputs:                                    # before the host-API leg below steps the same env again
        dump_outputs(args.dump_outputs, {"obs": env.obs, "reward": env.reward, "done": env.done, "info": env.info}, "" if world == 1 else "_rank%d" % rank)

    # end to end through the host-facing API: pinned H2D of the actions + step + D2H of obs/reward/done every step
    host_acts = np.random.default_rng(1234 + rank).uniform(-0.3, 0.3, (16, n, 12)).astype(np.float32)
    for k in range(5):
        env.step_host(host_acts[k % 16], info=True)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    Ke = min(K, 200)
    # wall-clock timing on a shared host: the run is cut into five blocks and the MEDIAN block rate is reported (every block rate goes into the
    # JSON line), so that one noisy-neighbour burst on the host cores does not decide the number
    NBLK = 5
    blk = max(1, Ke // NBLK); Ke = blk * NBLK
    blk_s = []
    for j in range(NBLK):
        t0 = time.perf_counter()
        for k in range(blk):
            env.step_host(host_acts[(j * blk + k) % 16], info=True)  # obs, reward, done AND the info rows train.py:150-157 reads every step
        torch.cuda.synchronize()
        blk_s.append(time.perf_counter() - t0)
    e2e_s = sorted(blk_s)[NBLK // 2] * NBLK
    e2e_blocks = [n * blk / t for t in blk_s]
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_val = world * n * Ke / float(te[0])
    clocks = sampler.stop() if rank == 0 else None
    env.close()
    extras = None
    if not args.no_extras:
        try:
            extras = run_extras(args, rank, world, local, dev, w, b)
        except Exception as ex:                                    # the headline line must survive a failing secondary measurement
            extras = {"error": repr(ex)}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs, peak_src = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json hbm_gbs)") if peaks.get("hbm_gbs") else (6650.0, "fallback")
        ms_per_step = total_ms / K
        achieved = ALG_BYTES_PER_ENV_STEP * n / (ms_per_step * 1e-3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_traffic.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
        # secondary (the bound that actually applies, SURVEY §8d): warp-instruction issue slots.  Instructions per launch are the
        # ncu count of the committed capture (profiles/step_kernel_r01e_ncu_full.csv); duration and SM clock are this run's.
        issue = None
        try:
            cands = sorted(f for f in os.listdir(os.path.join(ROOT, "profiles")) if f.startswith("step_kernel_r0") and f.endswith("_ncu_full.csv"))
            prof_name = cands[-1]
            prof = dict(l.split(",")[0::2] for l in open(os.path.join(ROOT, "profiles", prof_name)).read().splitlines()[2:] if l.count(",") == 2)
            inst = float(prof["smsp__inst_executed.sum"]) * n / 4096.0
            mhz = (clocks or {}).get("sm_mhz") or 1965.0
            slots = ms_per_step * 1e-3 * mhz * 1e6 * 148 * 4
            issue = {"warp_instructions_per_launch": inst, "issue_slot_frac": inst / slots, "fma_pipe_pct_ncu": float(prof["sm__pipe_fma_cycles_active.avg.pct_of_peak_sustained_active"]),
                     "warps_per_sm_ncu": float(prof["sm__warps_active.avg.per_cycle_active"]), "source": "profiles/" + prof_name}
        except Exception:
            pass
        cpu = None
        if not args.no_cpu_baseline:
            threads = host_threads()
            rate1, _ = cpu_oracle_rate(64, 8, 1, w, b)
            n_c = n                                                                        # the full 4096-env workload (same config as the GPU arm)
            steps_c = int(min(400, max(3, 12.0 * rate1 * threads / n_c)))                # ~12 s of CPU work at the ideal multi-thread rate
            rate, secs = cpu_oracle_rate(n_c, steps_c, threads, w, b)
            cpu = {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port", "per_thread": rate / threads, "single_thread": rate1,
                   "sample": "%d envs x %d control steps (%.1f s), float64 C oracle on %d pthreads; single-thread rate %.0f env-steps/s; NOT pybullet (absent)" % (n_c, steps_c, secs, threads, rate1)}
        line = {
            "metric": "env-steps/sec (A1, 4096 envs)", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "envs_per_gpu": n, "substeps_per_step": 13, "solver_iters": 23, "l2": "flushed between timed steps (256 MiB write outside the event pair)",
                       "timing": "per-step CUDA event pairs on the launching stream, max over ranks", "done_frac_last_step": done_frac},
            "e2e": {"value": e2e_val, "unit": "env-steps/s", "h2d_bytes_per_step": env.h2d_bytes_per_step(), "d2h_bytes_per_step": env.d2h_bytes_per_step(info=True), "steps": Ke, "estimator": "median of %d blocks of %d steps (wall clock)" % (NBLK, blk), "block_rates_rank0": e2e_blocks,
                    "transport": "numpy action -> pinned buffer -> step kernel reads it over PCIe and stores obs|reward|done and the info rows [N,56] (staged in shared memory, one coalesced block per CTA) straight to pinned host memory (b2q_step_host, B2Q_HOST_IO=2); stream sync every step"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs, "traffic": traffic,
                         "peak_source": peak_src, "kernel": "b2q_step_kernel<float>", "alg_bytes_per_env_step": ALG_BYTES_PER_ENV_STEP, "issue": issue,
                         "note": "latency/FP32-issue bound by construction (13 substeps x 23 PGS sweeps per launch on ~2.4 KB of state): HBM fraction is structurally tiny, see DESIGN.md §5"},
            "cpu_baseline": cpu,
            "clocks": clocks,
            "extras": extras,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
