"""Policy JSON import / export and batched evaluation.

Format and semantics follow the reference (paths relative to phoenix_drone_simulation/):
  utils/utils.py:362-430   dump_network_json: {"scaling_parameters": [mean[D], std[D]], "activation",
                           "0"/"1"/...: {"type": "standard", "weights": [out][in], "biases": [out]}}
  utils/utils.py:56-110    build_mlp_network(data): the loader used by load_network_json (:309-340)
  utils/evaluation.py:52-107  EnvironmentEvaluator: deterministic policy, one episode per evaluation,
                           returns / episode lengths / costs (`evaluate`: one policy, a host loop of policy and
                           env launches; `evaluate_many`: many policies on shared episodes, one kernel launch)
Only dense ("standard") layers are supported; the CSR product layers of the firmware export are not.
"""
import ctypes as C
import json

import numpy as np
import torch

from . import lib as _lib
from .config import EnvConfig
from .rollout import ActorCritic
from .vec_env import VecEnv


def export_policy_json(ac, path, activation='relu'):
    """Actor network + observation scaling of an ActorCritic -> JSON file (dump_network_json)."""
    lins = [m for m in ac.pi if isinstance(m, torch.nn.Linear)]
    d = lins[0].in_features
    mean = ac.obs_oms.mean if ac.obs_oms is not None else torch.zeros(d)
    std = ac.obs_oms.std if ac.obs_oms is not None else torch.ones(d)
    data = {'scaling_parameters': [mean.detach().cpu().double().tolist(), std.detach().cpu().double().tolist()],
            'activation': activation}
    for i, lin in enumerate(lins):
        data[str(i)] = {'type': 'standard', 'weights': lin.weight.detach().cpu().double().tolist(),
                        'biases': lin.bias.detach().cpu().double().tolist()}
    with open(path, 'w') as f:
        json.dump(data, f)
    return data


def load_policy_json(path, device='cuda', standardize=True, **ac_kwargs):
    """JSON file -> ActorCritic whose actor and observation scaling come from the file (the critic is
    freshly initialised: the export does not contain it).  Any two hidden layers of up to 64 units
    (experiments/05_impact_of_hidden_neurons trains 10 ... 64).  standardize=False drops the scaling:
    the network then sees raw observations, which is how the file's `check_sum` known answer is defined
    (utils/export.py:47-53: sum of net(ones)); `verify_check_sum` evaluates it."""
    with open(path) as f:
        data = json.load(f)
    layers = []
    while str(len(layers)) in data:
        entry = data[str(len(layers))]
        if entry.get('type', 'standard') != 'standard':
            raise NotImplementedError('only dense layers (type "standard") are supported')
        layers.append((torch.tensor(entry['weights'], dtype=torch.float32), torch.tensor(entry['biases'], dtype=torch.float32).reshape(-1)))
    if data.get('activation', 'relu') != 'relu' or len(layers) != 3:
        raise NotImplementedError('expected a relu actor with two hidden layers (ppo/defaults.py:6-19)')
    obs_dim, act_dim = layers[0][0].shape[1], layers[-1][0].shape[0]
    ac = ActorCritic(obs_dim, act_dim=act_dim, pi_hidden=(layers[0][0].shape[0], layers[1][0].shape[0]), device=device,
                     use_standardized_obs=standardize, **ac_kwargs)
    lins = [m for m in ac.pi if isinstance(m, torch.nn.Linear)]
    with torch.no_grad():
        for lin, (w, b) in zip(lins, layers):
            lin.weight.copy_(w)
            lin.bias.copy_(b)
        if standardize:
            sp = torch.tensor(data['scaling_parameters'], dtype=torch.float32)
            ac.obs_oms.mean.copy_(sp[0])
            ac.obs_oms.std.copy_(sp[1])
    ac.check_sum = float(data['check_sum']) if 'check_sum' in data else None
    return ac


@torch.no_grad()
def verify_check_sum(path, device='cuda', policy_kernel='tc', rtol=1e-5, atol=1e-5):
    """The reference's known-answer test for an exported policy (utils/export.py:47-53 writes it,
    utils/utils.py:324-330 is meant to check it): the sum of the network's outputs for an all-ones input
    must equal the file's `check_sum`.  Evaluated with the fused policy kernel selected by
    `policy_kernel` on CUDA devices (the torch modules on CPU).  Returns (got, expected)."""
    ac = load_policy_json(path, device=device, standardize=False, policy_kernel=policy_kernel)
    if ac.check_sum is None:
        raise ValueError(f'{path} carries no check_sum')
    d = ac.pi.net[0].in_features
    ones = torch.ones((128, d), dtype=torch.float32, device=device)       # one full tensor-core tile of identical rows
    if torch.device(device).type == 'cuda':
        n = ones.shape[0]
        act = torch.empty((n, 4), device=device); val = torch.empty(n, device=device)
        logp = torch.empty(n, device=device); mu = torch.empty((n, 4), device=device)
        ac.step_into(ones, act, val, logp, mu)
        assert bool((mu == mu[0]).all()), 'identical rows must give identical outputs'
        got = float(mu[0, :ac.log_std.shape[0]].double().sum())
    else:
        got = float(ac.pi(ones[:1]).double().sum())
    if abs(got - ac.check_sum) > atol + rtol * abs(ac.check_sum):
        raise AssertionError(f'check_sum mismatch: network gives {got}, file says {ac.check_sum}')
    return got, ac.check_sum


@torch.no_grad()
def evaluate(env_id, ac, num_evaluations=128, seed=0, device='cuda', **env_kwargs):
    """EnvironmentEvaluator.eval for `num_evaluations` episodes run in lock-step, one per environment,
    with the deterministic policy (action = mean, core.py:282-289).  Returns (returns, lengths, costs)."""
    env = VecEnv(env_id, num_evaluations, device=device, seed=seed, auto_reset=False, **env_kwargs)
    obs = env.reset()
    n = num_evaluations
    ret = torch.zeros(n, dtype=torch.float64, device=env.device)
    cost = torch.zeros(n, dtype=torch.float64, device=env.device)
    length = torch.zeros(n, dtype=torch.int64, device=env.device)
    alive = torch.ones(n, dtype=torch.bool, device=env.device)
    act = torch.empty((n, 4), dtype=torch.float32, device=env.device)
    val = torch.empty(n, dtype=torch.float32, device=env.device)
    logp = torch.empty(n, dtype=torch.float32, device=env.device)
    mu = torch.empty((n, 4), dtype=torch.float32, device=env.device)
    for _ in range(env.max_episode_steps):
        ac.step_into(obs.float().contiguous(), act, val, logp, mu)
        obs, r, term, trunc, info = env.step(mu)
        ret += r.double() * alive
        cost += info['cost'].double() * alive
        length += alive
        alive &= ~(term | trunc)
        if not bool(alive.any()):
            break
    return ret.cpu().numpy(), length.cpu().numpy(), cost.cpu().numpy()


def _actor_shape(ac):
    lins = [m for m in ac.pi if isinstance(m, torch.nn.Linear)]
    if len(lins) != 3:
        raise ValueError('evaluate_many needs actors with two hidden layers')
    return lins[0].in_features, (lins[0].out_features, lins[1].out_features), lins[2].out_features


def _check_policy_set(policies):
    """(obs_dim, pi_hidden, n_out, standardised, eps) shared by all `policies`; ValueError if they cannot share a
    launch.  Needs no device."""
    policies = list(policies)
    if not policies:
        raise ValueError('evaluate_many needs at least one policy')
    shapes = {_actor_shape(ac) for ac in policies}
    if len(shapes) != 1:
        raise ValueError(f'all policies must have the same obs_dim, pi_hidden and act_dim, got {sorted(shapes)}')
    obs_dim, hidden, n_out = shapes.pop()
    if max(hidden) > 64 or n_out > 4:
        raise ValueError(f'actor hidden sizes must be <= 64 and act_dim <= 4, got {hidden}, {n_out}')
    stdz = {ac.obs_oms is not None for ac in policies}
    if len(stdz) != 1:
        raise ValueError('either every policy standardises its observations (obs_oms) or none does')
    stdz = stdz.pop()
    eps = {float(ac.obs_oms.eps) for ac in policies} if stdz else {0.0}
    if len(eps) != 1:
        raise ValueError(f'all observation normalisers must use the same epsilon, got {sorted(eps)}')
    return obs_dim, hidden, n_out, stdz, eps.pop()


@torch.no_grad()
def _evaluate_many(env_id, policies, num_evaluations, seed, device, record, env_kwargs):
    policies = list(policies)
    obs_dim, hidden, n_out, stdz, eps = _check_policy_set(policies)
    P, E = len(policies), int(num_evaluations)
    if E < 1 or P * E >= 1 << 31:
        raise ValueError('num_evaluations must be >= 1 and len(policies) * num_evaluations < 2^31')
    kw = {k: v for k, v in env_kwargs.items() if k not in ('dtype', 'rng', 'env_offset', 'keep_final_obs')}
    env_dim = int((kw.get('config') or EnvConfig(env_id, **kw)).to_pdx().obs_dim)
    if env_dim != obs_dim:
        raise ValueError(f'the policies take obs_dim {obs_dim}, {env_id} with these options has {env_dim}')
    env_kwargs = dict(env_kwargs, auto_reset=False)
    env = VecEnv(env_id, E, device=device, seed=seed, **env_kwargs)
    dev = env.device
    L = env.lib
    for ac in policies:
        if any(p_.device != dev for p_ in ac.parameters()):
            raise ValueError(f'every policy must live on {dev}')
    st = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    # one pdx_policy_pack image per policy (the kernel reads the actor part)
    mlps = [(policies[0]._mlp_struct(ac.pi, n_out), policies[0]._mlp_struct(ac.v, 1)) for ac in policies]
    words = int(L.pdx_policy_pack_words(obs_dim, C.byref(mlps[0][0]), C.byref(mlps[0][1])))
    if words < 0:
        _lib.check(words)
    packed = torch.empty((P, words), dtype=torch.float32, device=dev)
    for k, (pi, v) in enumerate(mlps):
        _lib.check(L.pdx_policy_pack(obs_dim, C.byref(pi), C.byref(v), C.c_void_p(packed[k].data_ptr()), st))
    mean = std = None
    if stdz:
        mean = torch.stack([ac.obs_oms.mean.float() for ac in policies]).contiguous()
        std = torch.stack([ac.obs_oms.std.float() for ac in policies]).contiguous()
    # the episodes every policy shares: one reset of E environments, replicated per policy
    obs0 = env.reset()
    state = env.state.unsqueeze(0).repeat(P, 1, 1, 1)
    buf = _lib.PdxBuffers.from_buffer_copy(env._buf)
    buf.state, buf.obs = state.data_ptr(), obs0.data_ptr()
    s = _lib.PdxPolicySet()
    s.n_policies, s.episodes, s.obs_dim, s.n_out = P, E, obs_dim, n_out
    s.hidden[0], s.hidden[1] = hidden
    s.stride, s.packed = words, packed.data_ptr()
    s.mean = mean.data_ptr() if stdz else None
    s.std = std.data_ptr() if stdz else None
    s.eps = eps
    ret = torch.empty((P, E), dtype=torch.float64, device=dev)
    cost = torch.empty((P, E), dtype=torch.float64, device=dev)
    length = torch.empty((P, E), dtype=torch.int32, device=dev)
    out = _lib.PdxEvaluation()
    out.ret, out.cost, out.length = ret.data_ptr(), cost.data_ptr(), length.data_ptr()
    rec = None
    if record:
        T = env.max_episode_steps
        rec = {'obs': torch.full((T, P, E, obs_dim), float('nan'), device=dev),
               'act': torch.full((T, P, E, 4), float('nan'), device=dev),
               'reward': torch.full((T, P, E), float('nan'), device=dev),
               'cost': torch.full((T, P, E), float('nan'), device=dev),
               'terminated': torch.zeros((T, P, E), dtype=torch.uint8, device=dev),
               'truncated': torch.zeros((T, P, E), dtype=torch.uint8, device=dev)}
        for k in rec:
            setattr(out, 'rec_' + k, rec[k].data_ptr())
    # step t draws at counter + t: the counters `evaluate`'s VecEnv.step calls use after the same reset
    _lib.check(L.pdx_evaluate(C.byref(env.pdx), C.byref(buf), C.byref(s), C.byref(out), env.seed, env._counter + 1, st))
    result = (ret.cpu().numpy(), length.cpu().numpy().astype(np.int64), cost.cpu().numpy())
    return result + (rec,) if record else result


def evaluate_many(env_id, policies, num_evaluations=128, seed=0, device='cuda', **env_kwargs):
    """`evaluate` for a list of ActorCritic policies in one kernel launch (pdx_evaluate).  Episode e of every
    policy sees the same initial state and draws as episode e of `evaluate(env_id, ac, num_evaluations, seed)`,
    so a policy's results do not depend on the other policies of the call.  The action is the actor mean of
    the standardised observation, computed with the arithmetic of the CUDA-core policy kernel
    (ActorCritic(policy_kernel='cuda')).  All policies need the same obs_dim and pi_hidden and either all or
    none standardise observations (ValueError otherwise); float32 environments with Philox draws only.
    Returns (returns [P, E] float64, lengths [P, E] int64, costs [P, E] float64) as numpy arrays."""
    return _evaluate_many(env_id, policies, num_evaluations, seed, device, False, env_kwargs)
