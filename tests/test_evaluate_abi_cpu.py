"""pdx_evaluate's argument checks at the C ABI and evaluate_many's policy-set checks: both reject bad input before
any device call, and without a CUDA device a valid call fails with PDX_ERR_NO_DEVICE (there is no CPU path)."""
import ctypes as C

import pytest
import torch

import phoenix_drone_simulation_b200 as pds
from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.policy_io import evaluate_many
from phoenix_drone_simulation_b200.rollout import ActorCritic

PDX_ERR_INVALID, PDX_ERR_NO_DEVICE = -1, -3
FAKE = 0x1000          # never dereferenced: every check below happens before the library touches memory


@pytest.fixture(scope='module')
def lib():
    import os
    if not os.path.exists(L.LIB_PATH):
        from phoenix_drone_simulation_b200.build import build
        build()
    return L.load()


def _args(env_id='DroneHoverSimpleEnv-v0', P=3, E=128, **kw):
    cfg = pds.EnvConfig(env_id, **kw).to_pdx()
    buf = L.PdxBuffers()
    buf.n_envs, buf.device, buf.state, buf.obs = E, 0, FAKE, FAKE
    s = L.PdxPolicySet()
    s.n_policies, s.episodes, s.obs_dim, s.n_out = P, E, cfg.obs_dim, 4
    s.hidden[0], s.hidden[1] = 50, 50
    s.stride = 32 * 1024
    s.packed, s.mean, s.std, s.eps = FAKE, FAKE, FAKE, 1e-5
    out = L.PdxEvaluation()
    out.ret, out.cost, out.length = FAKE, FAKE, FAKE
    return cfg, buf, s, out


def _call(lib, cfg, buf, s, out):
    return lib.pdx_evaluate(C.byref(cfg) if cfg is not None else None, C.byref(buf) if buf is not None else None,
                            C.byref(s) if s is not None else None, C.byref(out) if out is not None else None, 0, 2, None)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
def test_valid_call_without_device_reports_no_device(lib):
    assert _call(lib, *_args()) == PDX_ERR_NO_DEVICE
    assert _call(lib, *_args('DroneTakeOffBulletEnv-v0', P=1, E=1, observation_history_size=16)) == PDX_ERR_NO_DEVICE


@pytest.mark.parametrize('which', ['cfg', 'buf', 'set', 'out'])
def test_null_arguments_are_invalid(lib, which):
    a = list(_args())
    a[['cfg', 'buf', 'set', 'out'].index(which)] = None
    assert _call(lib, *a) == PDX_ERR_INVALID


def _bad(name):
    def f(cfg, buf, s, out):
        if name == 'float64': cfg.dtype = L.PDX_DTYPE_F64
        elif name == 'tape': cfg.rng_mode = L.PDX_RNG_TAPE
        elif name == 'no_policies': s.n_policies = 0
        elif name == 'no_episodes': s.episodes = 0; buf.n_envs = 0
        elif name == 'too_many': s.n_policies = 1 << 16; s.episodes = 1 << 15; buf.n_envs = 1 << 15
        elif name == 'episodes_vs_n_envs': buf.n_envs = 127
        elif name == 'hidden_65': s.hidden[1] = 65
        elif name == 'hidden_0': s.hidden[0] = 0
        elif name == 'n_out_5': s.n_out = 5
        elif name == 'obs_dim': s.obs_dim = 35
        elif name == 'stride_short': s.stride = 100
        elif name == 'stride_unaligned': s.stride = 32 * 1024 + 1
        elif name == 'mean_without_std': s.std = None
        elif name == 'no_packed': s.packed = None
        elif name == 'no_state': buf.state = None
        elif name == 'no_obs0': buf.obs = None
        elif name == 'no_length': out.length = None
        elif name == 'partial_records': out.rec_obs = FAKE
        elif name == 'bad_config': cfg.history = 17
    return f


@pytest.mark.parametrize('name', ['float64', 'tape', 'no_policies', 'no_episodes', 'too_many', 'episodes_vs_n_envs',
                                  'hidden_65', 'hidden_0', 'n_out_5', 'obs_dim', 'stride_short', 'stride_unaligned',
                                  'mean_without_std', 'no_packed', 'no_state', 'no_obs0', 'no_length',
                                  'partial_records', 'bad_config'])
def test_out_of_range_arguments_are_invalid(lib, name):
    a = _args()
    _bad(name)(*a)
    assert _call(lib, *a) == PDX_ERR_INVALID, name
    assert lib.pdx_last_error().decode()


def test_all_record_buffers_are_accepted_as_a_set(lib):
    if torch.cuda.is_available():
        pytest.skip('the valid call would reach the device with fake pointers')
    cfg, buf, s, out = _args()
    for k in ('rec_obs', 'rec_act', 'rec_reward', 'rec_cost', 'rec_terminated', 'rec_truncated'):
        setattr(out, k, FAKE)
    assert _call(lib, cfg, buf, s, out) == PDX_ERR_NO_DEVICE


def _ac(obs_dim=34, hidden=(50, 50), stdz=True):
    return ActorCritic(obs_dim, pi_hidden=hidden, device='cpu', use_standardized_obs=stdz, policy_kernel='cuda')


@pytest.mark.parametrize('policies,match', [
    (lambda: [_ac(), _ac(hidden=(64, 64))], 'same obs_dim'),
    (lambda: [_ac(), _ac(stdz=False)], 'standardises'),
    (lambda: [_ac(), _ac(obs_dim=40)], 'same obs_dim'),
    (lambda: [_ac(obs_dim=40), _ac(obs_dim=40)], 'obs_dim 40'),
    (lambda: [], 'at least one'),
])
def test_policy_set_checks_raise_before_any_device_call(lib, policies, match):
    """device='cpu' would fail at VecEnv: the ValueError must come first."""
    with pytest.raises(ValueError, match=match):
        evaluate_many('DroneHoverSimpleEnv-v0', policies(), num_evaluations=8, device='cpu')


def test_episode_count_is_checked_before_any_device_call(lib):
    with pytest.raises(ValueError, match='num_evaluations'):
        evaluate_many('DroneHoverSimpleEnv-v0', [_ac()], num_evaluations=0, device='cpu')
