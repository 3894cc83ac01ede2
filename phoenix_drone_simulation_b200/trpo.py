"""TRPO on the batched engine: NPG's step direction with a backtracking line search (algs/trpo/trpo.py:8-64).

The search tries theta_old + 0.8^j step for j = 0 .. 14 and accepts the first candidate whose full-batch surrogate
loss is finite, does not increase and keeps the reference-normalised KL (npg.KL_SCALE) within 1.5 target_kl, the loss
improvement and the KL averaged across ranks.  With update_kernel='cuda' each candidate is one forward-only
pdx_ppo_pi_grad launch.
"""
import math

from .npg import NPG


def line_search(evaluate, step, theta_old, target_kl, total_steps=15, decay=0.8):
    """trpo.py search_step_size.  evaluate(theta) -> (loss_before - loss, kl), averaged across ranks.  Returns
    (step to add to theta_old, accept_step): accept_step j + 1 for candidate j, and (0 * step, 0) when none passes."""
    frac = 1.0
    for j in range(total_steps):
        improve, kl = evaluate(theta_old + frac * step)
        if math.isfinite(improve) and improve >= 0 and kl <= 1.5 * target_kl:
            return frac * step, j + 1
        frac *= decay
    return 0.0 * step, 0


class TRPO(NPG):
    def search_step_size(self, step, theta_old, evaluate):
        return line_search(evaluate, step, theta_old, self.target_kl)


def learn(env_id, **kwargs):
    """Counterpart of algs/trpo/trpo.py `learn(env_id, **kwargs) -> (ac, env)`."""
    return TRPO(env_id, **kwargs).learn()
