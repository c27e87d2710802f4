#!/usr/bin/env python
"""Time the UNMODIFIED reference (OpenRL, installed into oracle/_ref by oracle/make_ref.py) on the
host cores: `PPOAgent.train` through the reference's own public API and stock code path.

TEST / BENCH INFRASTRUCTURE (the reference arm of bench.py and the cpu_baseline leg).  Nothing of
openrl_b200 is on this path.  The third-party packages the reference imports and this image lacks
(gymnasium, treevalue, jsonargparse, ...) are the stand-ins under oracle/refstubs; CartPole-v1
dynamics come from oracle/cartpole_ref.py (gymnasium itself is absent — SURVEY.md §8c).

Protocol (SURVEY.md §8d, BASELINE.md §3): `make(env_id, env_num=N, asynchronous=...)` -> `PPONet` ->
`PPOAgent.train(total_time_steps)`, device cpu, `--episode_length T --ppo_epoch E`; wall clock over
`iters` iterations after `warmup` iterations, construction excluded; the reference's own FPS log
(`openrl/envs/vec_env/vec_info/simple_vec_info.py:30`) is captured as a cross-check.

    python oracle/run_reference.py --env CartPole-v1 --envs 128 --iters 5 --warmup 2 [--async]
Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))


def ref_paths():
    ref = os.path.join(HERE, "_ref")
    if not os.path.isdir(os.path.join(ref, "openrl")):
        raise SystemExit("oracle/_ref/openrl missing: run `python oracle/make_ref.py` where the reference source is")
    return [os.path.join(HERE, "refstubs"), HERE, ref]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--env", default="CartPole-v1")
    ap.add_argument("--envs", type=int, default=8)
    ap.add_argument("--T", type=int, default=128)
    ap.add_argument("--epochs", type=int, default=4)
    ap.add_argument("--minibatch", type=int, default=1)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--async", dest="asynchronous", action="store_true")
    ap.add_argument("--threads", type=int, default=0, help="torch intra-op threads (0 = calibrate: the fastest of 1 / 4 / 8 / 16 / 32, capped at the core count)")
    ap.add_argument("--extra", default="", help="extra reference flags, space separated")
    a = ap.parse_args()

    # torchrun exports OMP_NUM_THREADS=1; the reference arm uses every host core it can
    ncores = os.cpu_count() or 1
    # "all the host threads it can use": on many-core hosts torch's default (every core) makes these tiny ops slower, so
    # with --threads 0 the first iterations try several counts and the fastest is kept for the warm-up and the timed run
    cands = sorted({c for c in (1, 4, 8, 16, 32, min(ncores, 32)) if c <= ncores}) if not a.threads else []   # > 32 threads only slows these tiny ops
    threads = a.threads or min(ncores, 32)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ["MKL_NUM_THREADS"] = str(threads)
    for p in reversed(ref_paths()):
        sys.path.insert(0, p)
    os.environ["PYTHONPATH"] = os.pathsep.join(ref_paths() + [os.environ.get("PYTHONPATH", "")])  # AsyncVectorEnv workers

    import torch

    torch.set_num_threads(threads)

    import openrl.runners.common  # noqa: F401  (first: avoids the circular import through utils/callbacks)
    from openrl.configs.config import create_config_parser
    from openrl.drivers.onpolicy_driver import OnPolicyDriver
    from openrl.envs.common import make
    from openrl.modules.common import PPONet
    from openrl.runners.common import PPOAgent

    flags = ["--seed", "0", "--episode_length", str(a.T), "--ppo_epoch", str(a.epochs), "--num_mini_batch", str(a.minibatch),
             "--log_interval", "1"] + a.extra.split()
    cfg = create_config_parser().parse_args(flags)
    env = make(a.env, env_num=a.envs, asynchronous=a.asynchronous)
    net = PPONet(env, cfg=cfg, device="cpu")
    agent = PPOAgent(net)

    # per-iteration wall-clock stamps taken around the reference's own inner loop (the reference is
    # not modified: the bound method is wrapped at run time, as oracle/gen_golden.py does)
    stamps = []
    orig_inner = OnPolicyDriver._inner_loop

    cal = {"i": 0, "t": time.perf_counter(), "dur": {}}

    def inner(self):
        if cal["i"] < len(cands):
            torch.set_num_threads(cands[cal["i"]])
            cal["t"] = time.perf_counter()
        r = orig_inner(self)
        now = time.perf_counter()
        if cal["i"] < len(cands):
            cal["dur"][cands[cal["i"]]] = now - cal["t"]
            cal["i"] += 1
            if cal["i"] == len(cands):
                torch.set_num_threads(min(cal["dur"], key=cal["dur"].get))
            return r
        stamps.append(now)
        return r

    OnPolicyDriver._inner_loop = inner
    fps_log = []

    class FpsTap:
        """duck-typed logger: records what the reference itself reports (FPS from simple_vec_info.py:30)"""

        def __getattr__(self, name):
            return lambda *aa, **kk: None

        def log_info(self, infos, step):
            if "FPS" in infos:
                fps_log.append(float(infos["FPS"]))

    total = a.T * a.envs * (a.iters + a.warmup + len(cands))
    t_start = time.perf_counter()
    try:
        agent.train(total_time_steps=total, logger=FpsTap())
    finally:
        OnPolicyDriver._inner_loop = orig_inner
    env.close()
    if len(stamps) < a.warmup + a.iters:
        raise SystemExit(f"reference ran {len(stamps)} timed-phase iterations, expected {a.warmup + a.iters}")
    # stamps[i] = end of post-calibration iteration i; the timed window is iterations [warmup, warmup + iters)
    dt = stamps[a.warmup + a.iters - 1] - stamps[a.warmup - 1] if a.warmup > 0 else stamps[a.iters - 1] - t_start
    print(json.dumps({
        "env": a.env, "envs": a.envs, "T": a.T, "epochs": a.epochs, "asynchronous": a.asynchronous, "iters": a.iters,
        "warmup": a.warmup, "seconds": dt, "env_steps_per_s": a.T * a.envs * a.iters / dt,
        "reference_fps_log_last": fps_log[-1] if fps_log else None, "torch_threads": torch.get_num_threads(),
        "host_cores": ncores, "thread_calibration_s_per_iteration": {str(k): round(v, 4) for k, v in cal["dur"].items()},
        "processes": (a.envs + 1) if a.asynchronous else 1,
    }))


if __name__ == "__main__":
    main()
