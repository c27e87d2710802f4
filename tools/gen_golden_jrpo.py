#!/usr/bin/env python
"""Record the JRPO golden traces (tests/golden/trace_mpe_jrpo*.npz) by EXECUTING THE UNMODIFIED REFERENCE.

TEST INFRASTRUCTURE, run where the reference's source is available (it is not needed by the tests):

    PYTHONPATH=oracle/refstubs:oracle:<reference checkout> python tools/gen_golden_jrpo.py [--out DIR]

It drives `oracle/gen_golden.py: gen_trace` (initial / per-iteration parameters, rollout buffer, returns, every
torch.randperm, the six scalars of every ppo_update, ValueNorm state) and adds what that recorder does not capture
for the joint-action loss: the normalised advantages handed to ReplayData.recurrent_generator_v3
(replay_data.py:425-551), recorded by wrapping that bound method at run time, as `it<i>/advantages`.
Recorded with oracle.TRACE_THREADS intra-op threads, like the other traces.
"""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

import gen_golden  # noqa: E402  (oracle/ on PYTHONPATH; imports the reference)
from openrl.buffers.replay_data import ReplayData  # noqa: E402
from openrl.drivers.onpolicy_driver import OnPolicyDriver  # noqa: E402

# examples/mpe/mpe_jrpo.yaml (use_joint_action_loss with use_recurrent_policy), ppo_epoch 2, 4 envs, 2 iterations
JRPO = ["--seed", "0", "--episode_length", "25", "--ppo_epoch", "2", "--lr", "7e-4", "--critic_lr", "7e-4",
        "--use_recurrent_policy", "true", "--use_joint_action_loss", "true", "--use_valuenorm", "true",
        "--use_adv_normalize", "true", "--log_interval", "1000"]
TRACES = {
    # default data_chunk_length 2: chunks over g = n*T + t straddle two envs; one minibatch
    "mpe_jrpo": JRPO,
    # chunks of 5, two minibatches: per-minibatch agent-0 ValueNorm moments and loss weights
    "mpe_jrpo_mb2": JRPO + ["--data_chunk_length", "5", "--num_mini_batch", "2"],
}


def gen_jrpo_trace(tag, flags):
    it = {"n": -1}
    advantages = {}
    orig_cr, orig_v3 = OnPolicyDriver.compute_returns, ReplayData.recurrent_generator_v3

    def compute_returns(self):   # once per iteration, before that iteration's update
        it["n"] += 1
        return orig_cr(self)

    def v3(self, adv, *a, **k):
        advantages.setdefault(it["n"], adv.copy())
        return orig_v3(self, adv, *a, **k)

    OnPolicyDriver.compute_returns, ReplayData.recurrent_generator_v3 = compute_returns, v3
    try:
        gen_golden.gen_trace("simple_spread", 4, flags, 2, tag)
    finally:
        OnPolicyDriver.compute_returns, ReplayData.recurrent_generator_v3 = orig_cr, orig_v3
    path = os.path.join(gen_golden.OUT, f"trace_{tag}.npz")
    rec = dict(np.load(path, allow_pickle=True))
    assert sorted(advantages) == list(range(int(rec["meta/iters"]))), sorted(advantages)
    for i, adv in advantages.items():
        rec[f"it{i}/advantages"] = adv
    np.savez_compressed(path, **rec)
    print("added advantages to", path)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="", choices=[""] + list(TRACES))
    ap.add_argument("--out", default=gen_golden.OUT)
    a = ap.parse_args()
    sys.path.insert(0, ROOT)
    from oracle import TRACE_THREADS

    torch.set_num_threads(TRACE_THREADS)
    gen_golden.OUT = a.out
    os.makedirs(a.out, exist_ok=True)
    for tag, flags in TRACES.items():
        if a.only in ("", tag):
            gen_jrpo_trace(tag, flags)


if __name__ == "__main__":
    main()
