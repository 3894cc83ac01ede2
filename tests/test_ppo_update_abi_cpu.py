"""pdx_ppo_pi_grad / pdx_ppo_v_grad / pdx_ppo_scratch_bytes at the C ABI: every bad argument or unsupported shape is
rejected before any device call, and without a CUDA device a valid call fails with PDX_ERR_NO_DEVICE (there is no CPU
path).  The Python layer rejects networks outside the kernels' plan with ValueError."""
import ctypes as C

import pytest
import torch

from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.ppo import PPO, check_update_kernel_plan, pi_loss_and_grad, v_loss_and_grad
from phoenix_drone_simulation_b200.rollout import ActorCritic

PDX_ERR_INVALID, PDX_ERR_NO_DEVICE = -1, -3
FAKE = 0x1000          # never dereferenced: every check below happens before the library touches memory
BIG = 1 << 30


@pytest.fixture(scope='module')
def lib():
    import os
    if not os.path.exists(L.LIB_PATH):
        from phoenix_drone_simulation_b200.build import build
        build()
    return L.load()


def _args(n=1000, obs_dim=34, hidden=(50, 50), n_out=4):
    b = L.PdxPpoBatch()
    b.n, b.obs_dim = n, obs_dim
    b.obs, b.act, b.adv, b.logp_old, b.target_v = FAKE, FAKE, FAKE, FAKE, FAKE
    m = L.PdxMlp()
    m.hidden[0], m.hidden[1], m.n_out = hidden[0], hidden[1], n_out
    g = L.PdxMlpGrad()
    for k in range(3):
        m.weight[k] = m.bias[k] = g.weight[k] = g.bias[k] = FAKE
    return {'b': b, 'm': m, 'g': g, 'log_std': FAKE, 'clip': 0.2, 'loss': FAKE, 'mu': None, 'mu_ref': None,
            'kl': None, 'scratch': FAKE, 'scratch_bytes': BIG}


def _pi(lib, a):
    return lib.pdx_ppo_pi_grad(C.byref(a['b']) if a['b'] is not None else None, C.byref(a['m']) if a['m'] is not None else None,
                               a['log_std'], a['clip'], C.byref(a['g']) if a['g'] is not None else None, a['loss'],
                               a['mu'], a['mu_ref'], a['kl'], a['scratch'], a['scratch_bytes'], None)


def _v(lib, a):
    return lib.pdx_ppo_v_grad(C.byref(a['b']) if a['b'] is not None else None, C.byref(a['m']) if a['m'] is not None else None,
                              C.byref(a['g']) if a['g'] is not None else None, a['loss'], a['scratch'],
                              a['scratch_bytes'], None)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
def test_valid_calls_without_device_report_no_device(lib):
    for kw in ({}, {'n': 1, 'obs_dim': 384, 'hidden': (64, 64)}, {'obs_dim': 37, 'hidden': (7, 33)}):
        a = _args(**kw)
        assert _pi(lib, a) == PDX_ERR_NO_DEVICE
        assert 'no CPU path' in lib.pdx_last_error().decode()
        a['g'] = None                                      # forward-only mode
        a['mu'], a['mu_ref'], a['kl'] = FAKE, FAKE, FAKE
        assert _pi(lib, a) == PDX_ERR_NO_DEVICE
        a = _args(n_out=1, **kw)
        a['b'].index = FAKE
        assert _v(lib, a) == PDX_ERR_NO_DEVICE
        assert 'no CPU path' in lib.pdx_last_error().decode()
    m = _args()['m']
    assert lib.pdx_ppo_scratch_bytes(0, 34, C.byref(m)) == PDX_ERR_NO_DEVICE


def _bad(name):
    def f(a):
        b, m = a['b'], a['m']
        if name == 'no_batch': a['b'] = None
        elif name == 'no_net': a['m'] = None
        elif name == 'n_0': b.n = 0
        elif name == 'n_negative': b.n = -5
        elif name == 'obs_dim_0': b.obs_dim = 0
        elif name == 'obs_dim_385': b.obs_dim = 385
        elif name == 'no_obs': b.obs = None
        elif name == 'hidden_65': m.hidden[1] = 65
        elif name == 'hidden_0': m.hidden[0] = 0
        elif name == 'n_out': m.n_out = 3
        elif name == 'no_weight': m.weight[1] = None
        elif name == 'no_bias': m.bias[2] = None
        elif name == 'partial_grad': a['g'].bias[0] = None
        elif name == 'no_loss': a['loss'] = None
        elif name == 'no_scratch': a['scratch'] = None
        elif name == 'scratch_small': a['scratch_bytes'] = 64
    return f


COMMON = ['no_batch', 'no_net', 'n_0', 'n_negative', 'obs_dim_0', 'obs_dim_385', 'no_obs', 'hidden_65', 'hidden_0',
          'n_out', 'no_weight', 'no_bias', 'partial_grad', 'no_loss', 'no_scratch', 'scratch_small']


@pytest.mark.parametrize('name', COMMON + ['no_act', 'no_adv', 'no_logp_old', 'no_log_std', 'mu_ref_without_kl',
                                           'kl_without_mu_ref', 'clip_negative', 'clip_nan'])
def test_actor_bad_arguments_are_invalid(lib, name):
    a = _args()
    _bad(name)(a)
    if name == 'no_act': a['b'].act = None
    elif name == 'no_adv': a['b'].adv = None
    elif name == 'no_logp_old': a['b'].logp_old = None
    elif name == 'no_log_std': a['log_std'] = None
    elif name == 'mu_ref_without_kl': a['mu_ref'] = FAKE
    elif name == 'kl_without_mu_ref': a['kl'] = FAKE
    elif name == 'clip_negative': a['clip'] = -0.1
    elif name == 'clip_nan': a['clip'] = float('nan')
    assert _pi(lib, a) == PDX_ERR_INVALID, name
    assert lib.pdx_last_error().decode()


@pytest.mark.parametrize('name', COMMON + ['no_target_v', 'no_grad'])
def test_critic_bad_arguments_are_invalid(lib, name):
    a = _args(n_out=1)
    _bad(name)(a)
    if name == 'n_out': a['m'].n_out = 4
    elif name == 'no_target_v': a['b'].target_v = None
    elif name == 'no_grad': a['g'] = None
    assert _v(lib, a) == PDX_ERR_INVALID, name
    assert lib.pdx_last_error().decode()


@pytest.mark.parametrize('obs_dim,hidden,n_out', [(0, (50, 50), 4), (385, (50, 50), 4), (34, (65, 50), 4),
                                                  (34, (50, 50), 2)])
def test_scratch_bytes_rejects_bad_shapes(lib, obs_dim, hidden, n_out):
    m = _args(hidden=hidden, n_out=n_out)['m']
    assert lib.pdx_ppo_scratch_bytes(0, obs_dim, C.byref(m)) == PDX_ERR_INVALID


@pytest.mark.parametrize('kw', [dict(pi_hidden=(65, 50)), dict(v_hidden=(64, 80)), dict(pi_hidden=(50, 50, 50)),
                                dict(act_dim=3), dict(obs_dim=385)])
def test_networks_outside_the_plan_raise_value_error(lib, kw):
    obs_dim = kw.pop('obs_dim', 34)
    ac = ActorCritic(obs_dim, device='cpu', **kw)
    with pytest.raises(ValueError, match='update_kernel=cuda'):
        check_update_kernel_plan(ac)
    obs = torch.zeros((8, obs_dim))
    with pytest.raises(ValueError):
        pi_loss_and_grad(ac, obs, torch.zeros((8, 4)), torch.zeros(8), torch.zeros(8), 0.2)
    with pytest.raises(ValueError):
        v_loss_and_grad(ac, obs, torch.zeros(8))


def test_cpu_tensors_raise_value_error(lib):
    ac = ActorCritic(34, device='cpu')
    with pytest.raises(ValueError, match='CUDA'):
        v_loss_and_grad(ac, torch.zeros((8, 34)), torch.zeros(8))


@pytest.mark.parametrize('kw,match', [(dict(update_kernel='cuda', device='cpu'), 'CUDA device'),
                                      (dict(update_kernel='triton'), 'update_kernel')])
def test_ppo_constructor_rejects_before_building_anything(lib, kw, match):
    with pytest.raises(ValueError, match=match):
        PPO('DroneHoverSimpleEnv-v0', num_envs=8, **kw)
