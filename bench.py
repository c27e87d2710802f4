#!/usr/bin/env python
"""bench.py — env-steps/sec (collect + update) of the CartPole-v1 PPO hot path on B200.

Workload (BASELINE.json configs[1]): CartPole-v1 PPO, 4096 parallel envs PER GPU (weak scaling),
MLP policy/critic, 128-step rollout, 4 PPO epochs, 1 minibatch, device-resident env.step + GAE +
ppo_update kernels.  A "step" is one iteration = 128 vec-env steps + critic pass + GAE + 4 updates
= 4096*128 env-steps per GPU.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # + the last timed iteration's outputs, DIR/*.npy
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference          # CPU restatement of the reference path (oracle port)

One JSON line on rank 0 (see the contract in the task statement).  Timing: CUDA events per
iteration on the launching stream, L2 flushed (256 MB write) between timed iterations, max over
ranks; clocks sampled with nvidia-smi during the timed region.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS, T, EPOCHS, MINIBATCH = 4096, 128, 4, 1
FLAGS = ["--seed", "0", "--episode_length", str(T), "--ppo_epoch", str(EPOCHS), "--num_mini_batch", str(MINIBATCH),
         "--log_interval", "1000000", "--log_each_episode", "false"]
WORKLOAD = f"CartPole-v1 PPO, {N_ENVS} envs/GPU, T={T}, {EPOCHS} epochs x {MINIBATCH} minibatch, MLP 64x64"
METRIC = "env-steps/sec (collect+update), CartPole-v1 PPO"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.lines, self.proc, self.index = [], None, index
        self.window = None   # (t0, t1) wall-clock bounds of the timed region

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        lines = self.lines
        scope = "process lifetime (sampler runs from before warm-up to after the timed region)"
        if self.window is not None:
            inside = [x for x in lines if self.window[0] <= x[0] <= self.window[1] + 0.05]
            if len(inside) >= 3:
                lines, scope = inside, "timed region"
        for _, ln in lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [x for x in sm if x > 0.5 * max(mx)] if mx else sm   # samples taken under load
        return {"sm_mhz": statistics.median(busy or sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "scope": scope, "reasons": sorted(reasons)}


WORKLOADS = {
    # BASELINE.json configs; "c2" is the configuration the metric is quoted on (the bench line), the rest are reported as extras
    "c2": dict(env="CartPole-v1", envs=N_ENVS, T=T, flags=FLAGS),
    "c1": dict(env="CartPole-v1", envs=8, T=T, flags=FLAGS),
    "target128": dict(env="CartPole-v1", envs=128, T=T, flags=FLAGS),   # north_star's 128-env target point
    "c4": dict(env="GridWorldSelfPlay", envs=N_ENVS, T=T, flags=FLAGS + ["--selfplay_save_freq", "2"]),   # configs[3]: 2-player GridWorld vs opponent pool
    "c3": dict(env="simple_spread", envs=2048, T=25,
               flags=["--seed", "0", "--episode_length", "25", "--lr", "7e-4", "--critic_lr", "7e-4", "--use_recurrent_policy", "true",
                      "--use_valuenorm", "true", "--use_adv_normalize", "true", "--log_interval", "1000000", "--log_each_episode", "false"]),
}


class SyntheticHostEnv:
    """BASELINE configs[4] stand-in (mujoco is absent, SURVEY.md §8c/d): host-stepped env with HalfCheetah's shapes —
    obs ~ N(0,1) (N,1,17), reward ~ N(0,1), done ~ Bernoulli(1/1000), Box(6) actions — numpy on the host cores."""

    def __init__(self, n, obs_dim=17, act_dim=6, seed=0):
        import numpy as np

        from openrl_b200 import spaces

        self.parallel_env_num, self.agent_num = n, 1
        self.observation_space = spaces.Box(-np.inf, np.inf, (obs_dim,), np.float32)
        self.action_space = spaces.Box(-1, 1, (act_dim,), np.float32)
        self.rng, self.obs_dim, self.np = np.random.default_rng(seed), obs_dim, np

    def reset(self, seed=None):
        return self.rng.standard_normal((self.parallel_env_num, 1, self.obs_dim)).astype(self.np.float32)

    def step(self, actions):
        return self.step_range(0, self.parallel_env_num, actions)

    def step_range(self, lo, hi, actions):
        n = hi - lo
        return (self.rng.standard_normal((n, 1, self.obs_dim)).astype(self.np.float32), self.rng.standard_normal((n, 1, 1)),
                self.rng.random((n, 1)) < 1e-3, [{} for _ in range(n)])


def build_agent(rank, world, workload="c2", envs=None, extra_flags=()):
    import torch

    from openrl_b200.configs.config import create_config_parser
    from openrl_b200.envs.common import make
    from openrl_b200.modules.common import PPONet
    from openrl_b200.runners.common import PPOAgent

    w = WORKLOADS[workload]
    n = w["envs"] if envs is None else envs
    cfg = create_config_parser().parse_args(list(w["flags"]) + list(extra_flags))
    cfg.quiet = True
    dev = f"cuda:{torch.cuda.current_device()}"
    env = make(w["env"], env_num=n, device=dev, env_index_offset=rank * n)
    net = PPONet(env, cfg=cfg, device=dev)
    return cfg, env, net, PPOAgent(net, rank=rank, world_size=world)


def make_driver(cfg, env, net, agent, rank, world):
    from openrl_b200.algorithms.ppo import PPOAlgorithm
    from openrl_b200.buffers import NormalReplayBuffer
    from openrl_b200.drivers.onpolicy_driver import OnPolicyDriver

    A = env.agent_num
    trainer = PPOAlgorithm(cfg, net.module, agent_num=A, device=net.device)
    buf = NormalReplayBuffer(cfg, A, env.observation_space, env.action_space, device=net.device)
    drv = OnPolicyDriver({"cfg": cfg, "num_agents": A, "run_dir": None, "envs": env, "device": net.device}, trainer, buf,
                         agent, rank=rank, world_size=world, logger=None, callback=None)
    drv.reset_and_buffer_init()
    return drv


def gae_roofline(flush, steps=10):
    """GAE kernel alone at the C2 config shape (L2 flushed per launch) and at a >= 1 GB shape."""
    import torch

    from openrl_b200 import lib

    L = lib.load()
    out = {}
    for tag, Tn, B in (("config", T, N_ENVS), ("1GB", 128, 1 << 21)):
        dev = torch.device("cuda")
        r = torch.randn(Tn, B, device=dev); vp = torch.randn(Tn + 1, B, device=dev)
        m = (torch.rand(Tn + 1, B, device=dev) > 0.01).float(); act = torch.ones(Tn + 1, B, device=dev)
        vn = torch.tensor([0.3, 2.0, 0.5], device=dev); ret = torch.empty(Tn + 1, B, device=dev)
        adv = torch.empty(Tn, B, device=dev); st = torch.empty(8, dtype=torch.float64, device=dev)
        s = torch.cuda.current_stream().cuda_stream
        call = lambda: lib.check(L.orl_gae(lib.ptr(r), lib.ptr(vp), lib.ptr(m), None, lib.ptr(act), lib.ptr(vp[Tn]), lib.ptr(vn),  # noqa: E731
                                           lib.ptr(ret), lib.ptr(adv), lib.ptr(st), Tn, B, 0.99, 0.95, 5, s), "gae")
        for _ in range(3):
            call()
        ts = []
        for _ in range(steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); call(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t = statistics.mean(ts)
        bytes_per_el = 24  # rewards, value_preds, masks, active_masks in; returns, advantages out
        out[tag] = {"T": Tn, "B": B, "bytes_per_element": bytes_per_el, "avg_s": t, "GBps": Tn * B * bytes_per_el / t / 1e9}
        del r, vp, m, act, ret, adv
    return out


DUMP_LIMIT_BYTES = 64 << 20


def iteration_outputs(drv):
    """What one `device_iteration` hands its caller, as host arrays: the rollout buffer it filled (observations, actions,
    log-probs, rewards, masks, value predictions, returns, advantages), the updated policy / critic parameters, the
    ValueNorm state and the six per-update means of the logged loss terms (`train_info`, as `read_train_info` forms them);
    all float32."""
    d, tr = drv.buffer.data, drv.trainer
    out = {name: getattr(d, name) for name in ("policy_obs", "actions", "action_log_probs", "rewards", "masks", "active_masks",
                                               "value_preds", "returns", "advantages")}
    out["policy_params"] = tr.algo_module.models["policy"].flat_params
    out["critic_params"] = tr.algo_module.models["critic"].flat_params
    out["value_norm_state"] = tr.algo_module.get_critic_value_normalizer().state
    out["train_info"] = tr.train_info / (tr.ppo_epoch * tr.num_mini_batch)
    out = {k: v.detach().float().cpu().numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES} byte limit")
    return out


def dump_outputs(outputs, directory):
    import numpy as np

    os.makedirs(directory, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(directory, f"{name}.npy"), a)


def time_iterations(drv, steps, warmup, flush, world, after_timed=None):
    """W untimed + K timed device iterations (collect + update) through `OnPolicyDriver.device_iteration` — one captured
    CUDA graph replay per iteration when eligible (the product's default), else ~25 launches — CUDA events per iteration
    on the launching stream, 256 MB L2 flush between timed iterations, max over ranks.  The per-phase times come from a
    separate short eager pass (events cannot be read inside a graph); `after_timed(drv)`, when given, runs between the
    timed iterations and that pass, while the driver still holds what the last timed iteration computed.
    Returns (seconds, phases_ms, launches, wall window)."""
    import torch
    import torch.distributed as dist

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warmup, 3)):
        drv.device_iteration()
    barrier()
    l0 = drv.gpu_launches + drv.trainer.gpu_launches
    events = []
    barrier()
    t0 = time.time()
    for _ in range(steps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        drv.device_iteration()
        e1.record()
        events.append((e0, e1))
    barrier()
    window = (t0, time.time())
    launches = drv.gpu_launches + drv.trainer.gpu_launches - l0
    total_s = sum(a.elapsed_time(b) for a, b in events) * 1e-3
    if after_timed is not None:
        after_timed(drv)
    # phases: eager pass
    drv.phase_events = []
    for _ in range(3):
        flush.zero_()
        drv.device_iteration()
    barrier()
    phases = {}
    for name, a, b in drv.phase_events:
        phases.setdefault(name, []).append(a.elapsed_time(b))
    drv.phase_events = None
    t = torch.tensor([total_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), {k: statistics.mean(v) for k, v in phases.items()}, launches, window


def time_e2e(rank, world, steps, workload="c2", envs=None, extra_flags=()):
    """The same metric through the public API: PPOAgent.train(total_time_steps), wall clock, host logging and the
    per-iteration D2H metric reads inside; max over ranks.  Returns (seconds, h2d bytes/step, d2h bytes/step)."""
    import torch
    import torch.distributed as dist

    from openrl_b200.utils.logger import Logger

    cfg, env, net, agent = build_agent(rank, world, workload, envs, extra_flags)
    cfg.log_interval = 1
    n, Tn = env.parallel_env_num, cfg.episode_length
    agent.train(total_time_steps=n * Tn * 3, logger=Logger(quiet=True))  # warm-up call
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    tr, dr = agent.driver.trainer, agent.driver
    h0, d0 = tr.h2d_bytes + dr.h2d_bytes + getattr(env, "h2d_bytes", 0), tr.d2h_bytes + dr.d2h_bytes + getattr(env, "d2h_bytes", 0)
    t0 = time.perf_counter()
    agent.train(total_time_steps=n * Tn * steps, logger=Logger(quiet=True))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tr, dr = agent.driver.trainer, agent.driver
    h1, d1 = tr.h2d_bytes + dr.h2d_bytes + getattr(env, "h2d_bytes", 0), tr.d2h_bytes + dr.d2h_bytes + getattr(env, "d2h_bytes", 0)
    return float(t.item()), (h1 - h0) / steps, (d1 - d0) / steps


def side_result(rank, world, flush, workload, steps, envs=None, extra_flags=(), e2e=True):
    """A compact measurement of another configuration / mode (same timing rules), for the `extras` block."""
    cfg, env, net, agent = build_agent(rank, world, workload, envs, extra_flags)
    drv = make_driver(cfg, env, net, agent, rank, world)
    n, Tn = env.parallel_env_num, cfg.episode_length
    sec, phases, launches, _ = time_iterations(drv, steps, 3, flush, world)
    out = {"workload": f"{WORKLOADS[workload]['env']}, {n} envs/GPU x {env.agent_num} agent(s), T={Tn}, {cfg.ppo_epoch} epochs x {cfg.num_mini_batch} minibatch"
                       + (" " + " ".join(extra_flags) if extra_flags else ""),
           "value": n * Tn * steps * world / sec, "unit": "env-steps/s", "ms_per_step": sec / steps * 1e3,
           "phases_ms": {k: round(v, 4) for k, v in phases.items()}, "gpu_launches": launches, "steps": steps,
           "cuda_graph": getattr(drv, "_graph", None) is not None,
           "update_kernel": "tcgen05 split-fp16" if drv.trainer.use_tensor_cores else ("GRU warp kernels (fp32)" if drv.trainer.recurrent else "fp32 FFMA")}
    del drv
    if e2e:
        es, h2d, d2h = time_e2e(rank, world, steps, workload, envs, extra_flags)
        out["e2e"] = {"value": n * Tn * steps * world / es, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h}
    return out


def c5_result(steps=3, grouped=True):
    """BASELINE configs[4] class: host env.step (numpy stand-in with HalfCheetah shapes), device act + buffer + GAE +
    update, Gaussian head; measured through PPOAgent.train (there is no device-only form of this path)."""
    import torch

    from openrl_b200.configs.config import create_config_parser
    from openrl_b200.envs.vec_env import HostVecEnv
    from openrl_b200.modules.common import PPONet
    from openrl_b200.runners.common import PPOAgent
    from openrl_b200.utils.logger import Logger

    n, Tn = 1024, T
    cfg = create_config_parser().parse_args(FLAGS + ["--host_env_groups", "true" if grouped else "false"])
    cfg.quiet = True
    host = SyntheticHostEnv(n)
    env = HostVecEnv(host)
    agent = PPOAgent(PPONet(env, cfg=cfg, device=f"cuda:{torch.cuda.current_device()}"))
    agent.train(total_time_steps=n * Tn * 1, logger=Logger(quiet=True))
    torch.cuda.synchronize()
    h0, d0 = env.h2d_bytes, env.d2h_bytes
    t0 = time.perf_counter()
    agent.train(total_time_steps=n * Tn * steps, logger=Logger(quiet=True))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    # the host env alone (its numpy step is the floor of this path)
    a = host.rng.standard_normal((n, 1, 6)).astype("float32")
    t1 = time.perf_counter()
    for _ in range(Tn):
        host.step(a)
    host_s = time.perf_counter() - t1
    return {"workload": f"host-stepped synthetic HalfCheetah shapes (obs 17, Box(6)), {n} envs, T={Tn}, {EPOCHS} epochs, Gaussian head",
            "e2e": {"value": n * Tn * steps / dt, "unit": "env-steps/s", "h2d_bytes_per_step": (env.h2d_bytes - h0) / steps,
                    "d2h_bytes_per_step": (env.d2h_bytes - d0) / steps},
            "ms_per_step": dt / steps * 1e3, "host_env_only_ms_per_step": host_s * 1e3, "steps": steps,
            "ingest": "two env groups in ping-pong (device work of one group overlaps host stepping of the other)" if grouped
                      else "one group, synchronous (act -> D2H -> env.step -> H2D per step)"}


def ncu_traffic():
    """dram bytes per launch of the GAE kernel from the committed ncu capture summary (profiles/), or None."""
    for name in ("r2_ncu_gae.json", "r1_ncu_gae.json"):
        p = os.path.join(ROOT, "profiles", name)
        if os.path.exists(p):
            d = json.load(open(p))
            return d.get("dram_bytes_per_launch"), f"ncu --set full, profiles/{name} (dram__bytes_read.sum + dram__bytes_write.sum)"
    return None, "no ncu capture summary under profiles/"


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))

    flush = torch.empty(256 * 1024 * 1024 // 4, device="cuda")  # 256 MB > 126 MB L2
    cfg, env, net, agent = build_agent(rank, world, "c2")
    drv = make_driver(cfg, env, net, agent, rank, world)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dump = None
    if args.dump_outputs and rank == 0:
        dump = lambda d: dump_outputs(iteration_outputs(d), args.dump_outputs)  # noqa: E731
    total_s, phases, launches, window = time_iterations(drv, args.steps, args.warmup, flush, world, after_timed=dump)
    sampler.window = window
    clocks = sampler.stop() if rank == 0 else None
    env_steps = N_ENVS * T * args.steps * world
    value = env_steps / total_s
    tc_update = drv.trainer.use_tensor_cores
    graphed = getattr(drv, "_graph", None) is not None
    peer_exchange = getattr(drv.trainer, "peer", None) is not None
    del drv

    print("[bench] main timed region done", file=sys.stderr, flush=True)
    e2e_s, h2d, d2h = time_e2e(rank, world, args.steps, "c2")
    print("[bench] e2e done", file=sys.stderr, flush=True)

    strong = None
    if world > 1:
        # strong scaling (SURVEY.md §8d): the GLOBAL env count held at 4096, 4096 / N envs per GPU
        per = N_ENVS // world
        cs, es, ns, ags = build_agent(rank, world, "c2", envs=per)
        ds = make_driver(cs, es, ns, ags, rank, world)
        ss, sph, sl, _ = time_iterations(ds, args.steps, args.warmup, flush, world)
        strong = {"scaling": "strong", "global_envs": N_ENVS, "envs_per_gpu": per, "value": N_ENVS * T * args.steps / ss, "unit": "env-steps/s",
                  "ms_per_step": ss / args.steps * 1e3, "phases_ms": {k: round(v, 4) for k, v in sph.items()}, "gpu_launches": sl}
        del ds

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    hbm_peak, how = peaks()
    gae = gae_roofline(flush)
    gae_in_step = phases.get("gae", 0.0) * 1e-3
    upd_s = phases.get("update", 0.0) * 1e-3
    flops_update = 53e3 * N_ENVS * T * EPOCHS  # fwd+bwd of both nets, SURVEY.md §8d
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    tensor_peak = pk.get("bf16_tflops", 1668.8)   # fp16 and bf16 dense MMAs run at the same rate
    traffic, traffic_src = ncu_traffic()

    extras = {}
    if world == 1 and not args.no_extras:
        def guarded(name, fn):
            if args.only_extra and name not in args.only_extra.split(","):
                return
            t_ = time.time()
            print(f"[bench] extra {name} ...", file=sys.stderr, flush=True)
            try:
                extras[name] = fn()
            except Exception as e:  # noqa: BLE001
                extras[name] = {"error": f"{type(e).__name__}: {str(e)[-300:]}"}
            print(f"[bench] extra {name} done in {time.time() - t_:.1f} s", file=sys.stderr, flush=True)
        # the same C2 workload with the fp32 FFMA update kernel, and in parity mode (reference-order CPU noise + randperm)
        guarded("c2_fp32_ffma_update", lambda: side_result(0, 1, flush, "c2", 5, extra_flags=["--use_tensor_cores", "false"], e2e=False))
        guarded("c2_parity_mode", lambda: side_result(0, 1, flush, "c2", 3, extra_flags=["--parity_mode", "true"], e2e=False))
        guarded("target_128_envs", lambda: side_result(0, 1, flush, "target128", 10))
        guarded("c1_8_envs", lambda: side_result(0, 1, flush, "c1", 10))
        guarded("c3_mpe_gru_2048x3", lambda: side_result(0, 1, flush, "c3", 3, e2e=False))
        guarded("c4_selfplay_gridworld_4096", lambda: side_result(0, 1, flush, "c4", 5, e2e=False))
        guarded("c5_host_env_1024", lambda: c5_result(3))
        guarded("c5_host_env_1024_synchronous_ingest", lambda: c5_result(3, grouped=False))
    print("[bench] cpu baseline ...", file=sys.stderr, flush=True)
    cpu = None if args.no_cpu_baseline else cpu_baseline_sample(n_envs=256, iters=1)
    out = {
        "metric": METRIC, "value": value, "unit": "env-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_s / args.steps * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 (nets, losses, Adam; the three 64x64 GEMM groups of the update run as split-fp16 tcgen05 MMAs with fp32 "
                 "accumulation = fp32-class accuracy, the mode the 1e-4 parity tests run in), f64 (CartPole state)",
        "data": "synthetic: device-resident CartPole-v1, random-init nets, seed 0",
        "config": {"workload": WORKLOAD, "global_envs": N_ENVS * world, "rollout_T": T, "parallelism": f"env-shard dp{world}",
                   "gradient_exchange": ("none (1 GPU)" if world == 1 else
                                         "NVLink peer-memory sum fused into the optimiser kernel (orl_ppo_apply_peer)" if peer_exchange
                                         else "all-reduce between orl_ppo_reduce and orl_ppo_apply (NCCL, or symmetric one-shot with ORL_SYMM_ALLREDUCE=1)"),
                   "l2": "256 MB L2 flush between timed iterations; inside an iteration the 25 MB buffer is re-read by design",
                   "sampling": "device Philox4x32 action sampling, whole-buffer minibatch without a permutation (chi-square / moment "
                               "tested, tests/test_sampling_cuda.py); the reference-order CPU-noise mode is extras.c2_parity_mode"},
        "gpu_launches": launches,
        "launch_mode": ("one CUDA graph replay per iteration (the captured graph holds the kernel launches counted in gpu_launches)"
                        if graphed else "eager launches"),
        "phases_ms": phases, "phases_note": "per-phase CUDA-event times from a separate eager (non-graph) pass of 3 iterations",
        "e2e": {"value": env_steps / e2e_s, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "PPOAgent.train(total_time_steps) incl. per-iteration logging reads; the env is device-resident (north_star), "
                       "so a step has no host inputs"},
        "roofline": {"bound": "hbm", "kernel": "gae_scan_kernel (orl_gae), >=1 GB shape, L2 flushed", "achieved": gae["1GB"]["GBps"],
                     "peak": hbm_peak, "peak_source": how, "unit": "GB/s", "frac": gae["1GB"]["GBps"] / hbm_peak,
                     "algorithmic_bytes_per_launch": 128 * (1 << 21) * 24,
                     "traffic": traffic, "traffic_source": traffic_src,
                     "config_shape": {**gae["config"], "frac": gae["config"]["GBps"] / hbm_peak,
                                      "in_step_avg_s": gae_in_step,
                                      "in_step_GBps": N_ENVS * T * 24 / max(gae_in_step, 1e-12) / 1e9}},
        "roofline_dominant": {"kernel": "ppo_fwdbwd_tc_kernel (tcgen05 kind::f16, split-fp16 operands, 2 CTAs/SM)" if tc_update else "ppo_fwdbwd_kernel (fp32 FFMA)",
                              "share_of_step": upd_s / max(total_s / args.steps, 1e-12),
                              "bound": "tensor" if tc_update else "fp32 pipe",
                              "avg_s_per_iteration": upd_s, "launches_per_iteration": EPOCHS * MINIBATCH,
                              "algorithmic_flop_per_row": 53e3, "achieved": flops_update / max(upd_s, 1e-12) / 1e12, "unit": "TFLOP/s",
                              "peak": tensor_peak if tc_update else fp32_peak,
                              "frac": flops_update / max(upd_s, 1e-12) / 1e12 / (tensor_peak if tc_update else fp32_peak),
                              "frac_of_fp32_pipe_peak": flops_update / max(upd_s, 1e-12) / 1e12 / fp32_peak,
                              "note": "algorithmic FLOPs (53 kFLOP/row, SURVEY.md 8d); the split issues 3 MMAs per product and M=128 "
                                      "tiles with unused lanes, so tensor-pipe activity is higher than this fraction (ncu, profiles/)"},
        "cpu_baseline": cpu,
        "clocks": clocks,
    }
    if strong is not None:
        out["strong_scaling"] = strong
    if extras:
        out["extras"] = extras
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def _best_cpu_threads(n_envs):
    """The port is Python-dispatch-bound: torch intra-op threads mostly add overhead on these tiny
    matrices.  Time one iteration at 1 thread and at the default count and keep the faster setting
    ("all the host threads it can use" = the count that makes it fastest)."""
    import torch

    from oracle import loop as oloop

    default = torch.get_num_threads()
    best, best_t = default, None
    for nt in sorted({1, min(default, 8), default}):
        torch.set_num_threads(nt)
        cfg = oloop.cfg_from_flags(" ".join(FLAGS))
        tr = oloop.Trainer(cfg, "CartPole-v1", n_envs)
        t0 = time.perf_counter()
        tr.iteration()
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline_sample(n_envs=256, iters=1):
    """cpu_baseline leg: the unmodified reference (`kind: reference`, oracle/_ref through
    oracle/run_reference.py, SyncVectorEnv, 128 of the 4096 envs, all host cores) with the oracle port
    (oracle/loop.py) timed beside it as a second, labelled number."""
    from oracle import loop as oloop

    threads = _best_cpu_threads(n_envs)
    cfg = oloop.cfg_from_flags(" ".join(FLAGS))
    tr = oloop.Trainer(cfg, "CartPole-v1", n_envs)
    tr.iteration()  # warm-up
    t0 = time.perf_counter()
    for _ in range(iters):
        tr.iteration()
    dt = time.perf_counter() - t0
    port = {"value": n_envs * T * iters / dt, "unit": "env-steps/s", "cores": threads, "kind": "port",
            "sample": f"{iters} iteration(s) of {n_envs} envs x T={T}, {EPOCHS} epochs (oracle/loop.py, torch-CPU + numpy)"}
    if not reference_available():
        return {**port, "note": "oracle/_ref missing: port only"}
    try:
        ref = reference_run(REF_ENVS, 5, 3)
    except Exception as e:  # noqa: BLE001
        return {**port, "note": f"reference run failed ({str(e)[-200:]}): port only"}
    return {"value": ref["env_steps_per_s"], "unit": "env-steps/s", "cores": ref["torch_threads"], "kind": "reference",
            "sample": f"5 PPOAgent.train iterations (after 3 warm-up) of {REF_ENVS} of the {N_ENVS} envs x T={T}, {EPOCHS} epochs; unmodified "
                      f"reference from oracle/_ref, SyncVectorEnv, {ref['host_cores']} host cores", "port": port}


def reference_run(envs, iters, warmup, asynchronous=False, timeout=300):
    """One timed run of the UNMODIFIED reference (oracle/_ref, oracle/run_reference.py) in a fresh
    process: `PPOAgent.train` on the host cores, all of them (the child resets torchrun's OMP_NUM_THREADS=1)."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "run_reference.py"), "--env", "CartPole-v1", "--envs", str(envs),
           "--T", str(T), "--epochs", str(EPOCHS), "--minibatch", str(MINIBATCH), "--iters", str(iters), "--warmup", str(warmup)]
    if asynchronous:
        cmd.append("--async")
    env = {k: v for k, v in os.environ.items() if k not in ("OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"reference run failed (rc {r.returncode}): {r.stderr[-800:]}")
    return json.loads(lines[-1])


def reference_available():
    return os.path.isfile(os.path.join(ROOT, "oracle", "_ref", "openrl", "__init__.py"))


REF_ENVS = 128   # north_star's target point; the reference's per-env Python loop makes cost linear in envs


def run_reference(args):
    """Reference arm: the unmodified reference through its own public API (`make` -> `PPONet` ->
    `PPOAgent.train`, SyncVectorEnv) on the box's host cores.  Each step = one iteration of a bounded
    sample (128 of the 4096 envs; a 4096-env reference iteration takes ~30 s); the AsyncVectorEnv
    ("SubprocVecEnv", one process per env) run and the oracle port are reported beside it."""
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    if rank != 0:
        return
    steps, warmup = args.steps, max(args.warmup, 3)
    base = {"impl": "reference", "metric": METRIC, "unit": "env-steps/s", "n_gpus": world, "steps": steps, "warmup": warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD}}
    if reference_available():
        sync = reference_run(REF_ENVS, steps, warmup, asynchronous=False)
        value, kind = sync["env_steps_per_s"], "reference"
        extra = {"sync_128": sync}
        try:   # the north_star's "SubprocVecEnv" path: 128 worker processes + the learner
            extra["async_128"] = reference_run(REF_ENVS, max(2, min(steps, 3)), 1, asynchronous=True)
        except Exception as e:  # noqa: BLE001
            extra["async_128"] = {"error": str(e)[-300:]}
        try:
            extra["sync_8_c1"] = reference_run(8, 5, 2, asynchronous=False)
            extra["async_8_c1"] = reference_run(8, 5, 2, asynchronous=True)
        except Exception as e:  # noqa: BLE001
            extra["c1"] = {"error": str(e)[-300:]}
        extra["not_run"] = "AsyncVectorEnv at 4096 envs = 4097 processes: infeasible on this host; Sync at 4096 envs is ~30 s/iteration"
        cores, sample = sync["torch_threads"], (f"each step = one PPOAgent.train iteration of {REF_ENVS} of the {N_ENVS} envs x T={T}, {EPOCHS} epochs, "
                                                 f"unmodified reference (oracle/_ref) + SyncVectorEnv, {sync['host_cores']} host cores")
        dt = sync["seconds"]
    else:
        from oracle import loop as oloop

        n_envs = 256
        threads = _best_cpu_threads(n_envs)
        cfg = oloop.cfg_from_flags(" ".join(FLAGS))
        tr = oloop.Trainer(cfg, "CartPole-v1", n_envs)
        for _ in range(warmup):
            tr.iteration()
        t0 = time.perf_counter()
        for _ in range(steps):
            tr.iteration()
        dt = time.perf_counter() - t0
        value, kind, cores, extra = n_envs * T * steps / dt, "port", threads, {"note": "oracle/_ref missing: oracle port timed instead"}
        sample = f"each step = one iteration of {n_envs} of the {N_ENVS} envs x T={T}, {EPOCHS} epochs (oracle/loop.py)"
    cb = {"value": value, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample}
    print(json.dumps({**base, "value": value, "ms_per_step": dt / steps * 1e3, "cpu_baseline": cb, "reference_runs": extra,
                      "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="development: skip the cpu_baseline leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the extras block (other configs / modes)")
    ap.add_argument("--only-extra", default="", help="development: comma-separated names of the extras to run")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed iteration computed (rank 0) as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
