"""Actor-critic network with the reference's architecture (agent_network.py:5-81), batched.

Layer names and shapes match the reference's ``Agent`` (conv1, conv2, fc1, fc2, action_head, value_head),
so ``CtfPolicy.load_state_dict(reference_agent.state_dict())`` works.  This is stock torch/cuDNN — the
policy is outside the hot path of this repo (SURVEY.md §2 row 6); it exists so the batched rollout / duel
adapters and BASELINE config 5 can run where the reference tree is absent.
For rollout / duel inference from packed observations use ``fused_policy.FusedPolicy`` (bf16, a CUDA trunk kernel).
"""
from __future__ import annotations

import torch
import torch.nn as nn
from torch.distributions.categorical import Categorical


class CtfPolicy(nn.Module):
    def __init__(self, n_actions, n_channels, grid_size, metadata_size, use_masking=True):
        super().__init__()
        self.n_actions, self.n_channels, self.grid_size, self.metadata_size = n_actions, n_channels, grid_size, metadata_size
        self.use_masking = use_masking
        side = grid_size - 4  # two valid 3x3 convolutions
        self.unrolled_conv_size = 32 * side * side
        self.conv1 = nn.Conv2d(n_channels, 16, kernel_size=3, stride=1)
        self.conv2 = nn.Conv2d(16, 32, kernel_size=3, stride=1)
        self.fc1 = nn.Linear(self.unrolled_conv_size + metadata_size, 256)
        self.fc2 = nn.Linear(256, 128)
        self.action_head = nn.Linear(128, n_actions)
        self.value_head = nn.Linear(128, 1)
        # agent types with AGENT_TYPE_ACTION_MASK == 1 may only use actions 0..4 (agent_network.py:21, 66-75)
        self.register_buffer("mask_5", torch.tensor([1.0] * 5 + [0.0] * (n_actions - 5)), persistent=False)

    def forward(self, grid, meta):
        x = torch.tanh(self.conv1(grid))
        x = torch.tanh(self.conv2(x))
        x = torch.cat((x.reshape(-1, self.unrolled_conv_size), meta), dim=1)
        x = torch.tanh(self.fc1(x))
        x = torch.tanh(self.fc2(x))
        return self.value_head(x), self.action_head(x)

    def masked_logits(self, logits, use_action_mask):
        if not self.use_masking:
            return logits
        m = use_action_mask.reshape(-1, 1)
        mask = torch.where(m == 1, self.mask_5.unsqueeze(0), torch.ones_like(logits))
        return logits + (mask - 1.0) * 1e9

    def get_action_and_value(self, grid, meta, use_action_mask, action=None):
        value, logits = self(grid, meta)
        probs = Categorical(logits=self.masked_logits(logits, use_action_mask), validate_args=False)
        if action is None:
            action = probs.sample()
        return action, probs.log_prob(action), probs.entropy(), value

    def get_action(self, grid, meta, use_action_mask):
        _, logits = self(grid, meta)
        # validate_args=False: the argument check reads a flag back to the host, which a CUDA graph capture forbids
        return Categorical(logits=self.masked_logits(logits, use_action_mask), validate_args=False).sample()

    def get_value(self, grid, meta):
        return self(grid, meta)[0]
