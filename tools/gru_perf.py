"""Phase timing of the recurrent (GRU) MAPPO path at BASELINE configs[2] shape: simple_spread, 3 agents x 2048 envs,
T=25, shared actor-critic GRU, default ppo_epoch (10), data_chunk_length 2 (examples/mpe/mpe_ppo.yaml).  Fast mode (device Philox).

    python tools/gru_perf.py [N [iters]] [--joint]

--joint also times the joint-action loss (JRPO, examples/mpe/mpe_jrpo.yaml) at the same shape, alternating with MAPPO-GRU;
each reports the best of three windows of `iters` iterations."""
import faulthandler, json, os, sys
faulthandler.dump_traceback_later(280, exit=True)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
from openrl_b200.configs.config import create_config_parser
from openrl_b200.envs.common import make
from openrl_b200.modules.common import PPONet
from openrl_b200.runners.common import PPOAgent
from openrl_b200.utils.logger import Logger

# --joint: the same shape with the joint-action loss (JRPO, examples/mpe/mpe_jrpo.yaml) timed against MAPPO-GRU in the same
# process, the two alternating over `rounds` windows so that host noise hits both alike
argv = [a for a in sys.argv[1:] if a != "--joint"]
joint = "--joint" in sys.argv[1:]
N = int(argv[0]) if len(argv) > 0 else 2048
iters = int(argv[1]) if len(argv) > 1 else 5
rounds = 3 if joint else 1


def make_driver(use_joint):
    cfg = create_config_parser().parse_args(["--episode_length", "25", "--lr", "7e-4", "--critic_lr", "7e-4", "--use_recurrent_policy", "true",
                                             "--use_valuenorm", "true", "--use_adv_normalize", "true",
                                             "--use_joint_action_loss", str(use_joint).lower()])
    cfg.quiet = True
    env = make("simple_spread", env_num=N)
    agent = PPOAgent(PPONet(env, cfg=cfg, device="cuda:0"))
    agent.train(total_time_steps=0, logger=Logger(quiet=True))
    drv = agent.driver
    for _ in range(2):
        drv.device_iteration()
    torch.cuda.synchronize()
    return cfg, drv


def window(drv):
    drv.phase_events = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        drv.device_iteration()
    e1.record()
    torch.cuda.synchronize()
    phases = {}
    for name, a, b in drv.phase_events:
        phases[name] = phases.get(name, 0.0) + a.elapsed_time(b) / iters
    return e0.elapsed_time(e1) / iters, phases


runs = {"mappo_gru": make_driver(False)}
if joint:
    runs["jrpo"] = make_driver(True)
res = {k: [] for k in runs}
for _ in range(rounds):
    for k, (cfg, drv) in runs.items():
        res[k].append(window(drv))
out = {}
for k, (cfg, drv) in runs.items():
    ms_all = [m for m, _ in res[k]]
    ms, phases = min(res[k], key=lambda r: r[0])
    out[k] = {"workload": f"simple_spread GRU {'JRPO' if cfg.use_joint_action_loss else 'MAPPO'} {N} envs x 3 agents, T=25, "
                          f"ppo_epoch {cfg.ppo_epoch}, L={cfg.data_chunk_length}",
              "ms_per_iter": round(ms, 3), "ms_per_iter_all_windows": [round(m, 3) for m in ms_all],
              "env_steps_per_s": round(N * 25 / (ms * 1e-3)),
              "phases_ms": {p: round(v, 3) for p, v in phases.items()}, "train_info": drv.trainer.read_train_info()}
out["device"] = torch.cuda.get_device_name(0)
try:
    import subprocess
    out["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                                        capture_output=True, text=True, timeout=30).stdout.strip()
except Exception as e:   # the timing stands without it; say that it is missing
    out["power_limit"] = f"unavailable ({e})"
print(json.dumps(out if joint else dict(out["mappo_gru"], device=out["device"], power_limit=out["power_limit"])))
