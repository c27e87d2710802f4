"""A2CAlgorithm (reference: openrl/algorithms/a2c.py:27-145): PPOAlgorithm with the policy loss
-adv * log-prob (a2c.py:88-98), one minibatch per epoch (a2c.py:37) and no `ratio` metric (a2c.py:142-145).
Same CUDA kernels, different loss epilogue (ORL_PPO_A2C)."""
from .. import lib
from .ppo import PPOAlgorithm


class A2CAlgorithm(PPOAlgorithm):
    def __init__(self, cfg, init_module, agent_num=1, device="cuda:0"):
        if getattr(cfg, "use_joint_action_loss", False):
            # the reference's A2C loss (a2c.py:39-140) has no joint-action branch
            raise NotImplementedError("use_joint_action_loss with A2C is not built")
        super().__init__(cfg, init_module, agent_num, device)
        self.num_mini_batch = 1
        self.flags |= lib.PPO_A2C

    def train(self, buffer, turn_on=True):
        info = super().train(buffer, turn_on)
        info.pop("ratio", None)
        return info
