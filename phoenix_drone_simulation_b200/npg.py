"""Natural policy gradient on the batched engine: PPO's rollout and value phase, a conjugate-gradient policy step.

Mirrors the reference (paths relative to phoenix_drone_simulation/):
  algs/npg/npg.py:15-182   NPGAlgorithm: Fvp on every 4th observation, update_policy_net (surrogate gradient g,
                           x = CG(F, -g), step = sqrt(2 target_kl / x^T F x) x), no pi optimiser and no schedule
  algs/utils.py:5-96       conjugate_gradients, flat parameters of ac.pi.net
The surrogate is IWPG's unclipped -(r A).mean().  With update_kernel='cuda' its gradient comes from pdx_ppo_pi_grad
(clip_ratio = inf) and every Fisher-vector product from pdx_ppo_pi_fvp; with 'torch' both are autograd (the Fvp is the
reference's double backward, ppo.pi_fvp_torch).

KL normalisation, decided here once: the reference's policy distribution is a per-dimension Normal, so its
kl_divergence(p, q).mean() averages over the 4 action dimensions as well as the samples.  pdx_ppo_pi_grad's kl sums
over the dimensions, so NPG / TRPO use kl / 4 (KL_SCALE) for the trust region and scale = 1/4 for the Fvp.  (PPO's
KL early stop uses the summed kl, 4x the reference's value.)
"""
import torch

from .ppo import PPO, pi_flat_params, pi_fvp, pi_fvp_torch, pi_loss_and_grad, pi_net_params, set_pi_flat_params
from .rollout import _world

KL_SCALE = 0.25          # the reference's per-dimension KL mean: 1 / act_dim of the summed Gaussian KL


def conjugate_gradients(Avp, b, nsteps, residual_tol=1e-10, eps=1e-6):
    """algs/utils.py conjugate_gradients: x ~ A^-1 b in at most `nsteps` products Avp(p).  The reference's first
    product Avp(0) is exactly zero and is skipped (r = b)."""
    x = torch.zeros_like(b)
    r = b.clone()
    p = r.clone()
    rdotr = torch.dot(r, r)
    for _ in range(nsteps):
        z = Avp(p)
        alpha = rdotr / (torch.dot(p, z) + eps)
        x += alpha * p
        r -= alpha * z
        new_rdotr = torch.dot(r, r)
        if torch.sqrt(new_rdotr) < residual_tol:
            break
        mu = new_rdotr / (rdotr + eps)
        p = r + mu * p
        rdotr = new_rdotr
    return x


class NPG(PPO):
    def __init__(self, env_id, cg_iters=10, cg_damping=0.1, target_kl=0.01, **kwargs):
        super().__init__(env_id, target_kl=target_kl, **kwargs)
        self.clip_ratio = None                               # the unclipped surrogate
        self.cg_iters, self.cg_damping = cg_iters, cg_damping
        self.sched = None                                    # npg.py: no pi optimiser step, scheduler = None
        self.step_info = {}

    def update(self, data):
        info = super().update(data)
        info.update(self.step_info)
        return info

    def _allreduce_mean(self, t):
        P = _world(self.dist)
        if P > 1:
            self.dist.all_reduce(t)
            t /= P
        return t

    def _surrogate_grad(self, obs, act, adv, logp_old):
        """(loss, flat gradient) of -(r A).mean() on the full batch, both averaged across ranks."""
        if self.update_kernel == 'cuda':
            loss, _ = pi_loss_and_grad(self.ac, obs, act, adv, logp_old, None)
        else:
            self.pi_opt.zero_grad(set_to_none=True)
            loss = self._loss_pi(obs, act, adv, logp_old)[0]
            loss.backward()
        self._avg_grads(self.ac.pi)
        g = torch.cat([p_.grad.reshape(-1) for p_ in pi_net_params(self.ac)])
        return self._allreduce_mean(loss.detach().reshape(1).clone())[0], g

    def _fvp(self, obs, idx, v):
        """F v averaged across ranks, plus cg_damping v (npg.py Fvp)."""
        if self.update_kernel == 'cuda':
            out = pi_fvp(self.ac, obs, v, self.cg_damping, KL_SCALE, index=idx)
        else:
            out = pi_fvp_torch(self.ac, obs, v, self.cg_damping, KL_SCALE, index=idx)
        return self._allreduce_mean(out)

    def _loss_kl(self, obs, act, adv, logp_old, mu_old):
        """Forward only: (surrogate loss, reference-normalised KL to mu_old) as device scalars, this rank only."""
        if self.update_kernel == 'cuda':
            mu = torch.empty_like(mu_old)
            loss, kl = pi_loss_and_grad(self.ac, obs, act, adv, logp_old, None, grad=False, mu=mu, mu_ref=mu_old)
            return loss, kl * KL_SCALE
        with torch.no_grad():
            loss = self._loss_pi(obs, act, adv, logp_old)[0]
            return loss, self._pi_forward(obs, act, adv, logp_old, mu_ref=mu_old)[1] * KL_SCALE

    def search_step_size(self, step, theta_old, evaluate):
        """NPG takes the whole natural-gradient step.  Returns (step to add, accept_step)."""
        return step, 1

    def update_pi(self, obs, act, adv, logp_old):
        """npg.py update_policy_net.  Returns (loss after the step, 0, kl after the step)."""
        if self.update_kernel == 'cuda':
            obs, act, adv, logp_old = obs.contiguous(), act.contiguous(), adv.contiguous(), logp_old.contiguous()
        fvp_idx = torch.arange(0, obs.shape[0], 4, device=obs.device)
        mu_old = self._pi_forward(obs, act, adv, logp_old)[0]
        theta_old = pi_flat_params(self.ac)
        loss_before, g = self._surrogate_grad(obs, act, adv, logp_old)
        x = conjugate_gradients(lambda v: self._fvp(obs, fvp_idx, v), -g, self.cg_iters)
        xHx = torch.dot(x, self._fvp(obs, fvp_idx, x))
        step = torch.sqrt(2 * self.target_kl / (xHx + 1e-8)) * x

        def evaluate(theta):
            """(loss improvement, kl) of the actor at theta, averaged across ranks, as host floats."""
            set_pi_flat_params(self.ac, theta)
            loss, kl = self._loss_kl(obs, act, adv, logp_old, mu_old)
            t = self._allreduce_mean(torch.stack([loss_before - loss, kl]))
            return float(t[0]), float(t[1])

        final_step, accept = self.search_step_size(step, theta_old, evaluate)
        set_pi_flat_params(self.ac, theta_old + final_step)
        loss, kl = self._loss_kl(obs, act, adv, logp_old, mu_old)
        kl = float(self._allreduce_mean(kl.reshape(1).clone()))
        self.step_info = {'accept_step': accept, 'xHx': float(xHx)}
        return loss, 0, kl


def learn(env_id, **kwargs):
    """Counterpart of algs/npg/npg.py `learn(env_id, **kwargs) -> (ac, env)`."""
    return NPG(env_id, **kwargs).learn()

