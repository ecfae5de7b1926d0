"""Policy containers with the reference's parameter layout.

Reference: rl_sde_is/models.py:4-18 (``mlp``) and reinforce_deterministic_core.py:13-28
(``DeterministicPolicy``).  The module is only a parameter container + a plain torch forward for
host-side use (plots, tests); the rollouts evaluate the policy inside the fused CUDA kernels, reading
the parameters in state_dict order: ``policy.0.weight (H,d)``, ``policy.0.bias (H)``,
``policy.2.weight (H,H)``, ``policy.2.bias (H)``, ``policy.4.weight (d,H)``, ``policy.4.bias (d)``.

``TabularPolicy`` is a 1-D control tabulated on ``env.state_space_h`` (the DP greedy policy, the HJB solution u*): the
rollouts of ``approximate_methods`` evaluate it inside their own kernel (``rlsde_rollout_fwd_table``).
"""
import numpy as np
import torch
import torch.nn as nn


def mlp(sizes, activation, output_activation=nn.Identity()):
    """Linear / activation stack; the last Linear is followed by ``output_activation``."""
    n = len(sizes) - 1
    stack = []
    for j, (fan_in, fan_out) in enumerate(zip(sizes[:-1], sizes[1:])):
        stack.append(nn.Linear(fan_in, fan_out))
        stack.append(output_activation if j == n - 1 else activation)
    return nn.Sequential(*stack)


class DeterministicPolicy(nn.Module):
    """a = mu_theta(x); head initialised U(-5e-3, 5e-3) so the initial control is ~0."""

    HEAD_INIT = 5e-3

    def __init__(self, state_dim, action_dim, hidden_sizes, activation):
        super().__init__()
        self.sizes = [state_dim, *hidden_sizes, action_dim]
        self.policy = mlp(sizes=self.sizes, activation=activation)
        # the reference re-initialises every Linear whose out_features equals the action dimension
        for layer in self.policy:
            if isinstance(layer, nn.Linear) and layer.out_features == self.sizes[-1]:
                nn.init.uniform_(layer.weight, -self.HEAD_INIT, self.HEAD_INIT)
                nn.init.uniform_(layer.bias, -self.HEAD_INIT, self.HEAD_INIT)

    def forward(self, state):
        return self.policy(state)


class TabularPolicy(nn.Module):
    """u(x) = actions[idx(x)] on the 1-D state grid ``env.state_space_h``, with the index of
    ``env.get_state_idx_truncate``: idx(x) = floor((clip(x, low, high) - low) / h_state), computed in float64 and clamped
    to the table.  The GPU rollouts evaluate the same lookup on the state in state precision.

    ``actions``: shape (n_states, 1) or (n_states,), e.g. ``env.action_space_h[greedy_action_idx]`` (DP) or ``sol.policy_opt_table(env)``
    (HJB).  The table is a float32 buffer, not a parameter: a TabularPolicy cannot be trained."""

    def __init__(self, env, actions):
        super().__init__()
        if int(env.d) != 1:
            raise ValueError(f"a TabularPolicy is a control on the 1-D state grid; env.d = {env.d}")
        a = torch.as_tensor(np.asarray(actions.detach().cpu() if torch.is_tensor(actions) else actions, dtype=np.float32))
        n = int(env.n_states)
        if tuple(a.shape) not in ((n, 1), (n,)):
            raise ValueError(f"actions must have shape ({n}, 1) or ({n},) (env.state_space_h), got {tuple(a.shape)}")
        self.register_buffer("table", a.reshape(n, 1).clone())
        self.low, self.high, self.h = float(env.state_space_low), float(env.state_space_high), float(env.h_state)

    @property
    def grid(self):
        """``(low, high, h)`` of the state grid the table lives on."""
        return self.low, self.high, self.h

    def index(self, state):
        """idx(x) of every row of ``state`` (shape (..., 1)), int64, clamped to [0, n_states - 1]."""
        x = torch.as_tensor(state).detach().to(device=self.table.device, dtype=torch.float64)[..., 0]
        gi = torch.floor((x.clamp(self.low, self.high) - self.low) / self.h).long()
        return gi.clamp(0, self.table.shape[0] - 1)

    def forward(self, state):
        return self.table[self.index(state)]
