"""The population entry points (pdx_policy_step_members, pdx_gae_members, pdx_moments_members,
pdx_ppo_pi_grad_members, pdx_ppo_v_grad_members, pdx_adam_members) reject bad arguments with PDX_ERR_INVALID before any device call,
and PopulationPPO rejects what it cannot run before it touches a device."""
import ctypes as C
import os

import pytest

from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.population import PopulationPPO

PDX_ERR_INVALID = -1
FAKE = 0x1000          # never dereferenced: every check below happens before the library touches memory
BIG = 1 << 40


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(L.LIB_PATH):
        from phoenix_drone_simulation_b200.build import build
        build()
    return L.load()


def test_abi_version(lib):
    assert L.ABI_VERSION == 8
    assert lib.pdx_abi_version() == L.ABI_VERSION


def _mlp(hidden=(50, 50), n_out=4):
    m = L.PdxMlp()
    m.hidden[0], m.hidden[1], m.n_out = hidden[0], hidden[1], n_out
    for k in range(3):
        m.weight[k] = m.bias[k] = FAKE
    return m


# ---- pdx_policy_step_members -----------------------------------------------------------------------
def _policy(lib, P=3, n=1000, obs_dim=34, pi=None, v=None, stride=None, obs=FAKE, packed=FAKE, mean=FAKE, std=FAKE,
            act=FAKE):
    pi = pi or _mlp()
    v = v or _mlp((64, 64), 1)
    if stride is None:
        stride = int(lib.pdx_policy_pack_words(min(obs_dim, 384), C.byref(_mlp()), C.byref(_mlp((64, 64), 1))))
    return lib.pdx_policy_step_members(P, n, obs_dim, obs, mean, std, 1e-5, C.byref(pi), C.byref(v), FAKE, packed,
                                       stride, 0, 1, 0, act, FAKE, FAKE, None, None)


@pytest.mark.parametrize('case', [
    dict(P=0), dict(P=-1), dict(P=65536), dict(n=0), dict(obs_dim=0), dict(obs_dim=385),
    dict(obs=None), dict(packed=None), dict(act=None), dict(mean=None), dict(std=None),
    dict(pi=_mlp((65, 50))), dict(pi=_mlp((50, 65))), dict(v=_mlp((64, 65), 1)), dict(pi=_mlp(n_out=5)),
    dict(stride=10), dict(stride=-4),
])
def test_policy_step_members_rejects(lib, case):
    assert _policy(lib, **case) == PDX_ERR_INVALID


def test_policy_step_members_rejects_misaligned_stride(lib):
    words = int(lib.pdx_policy_pack_words(34, C.byref(_mlp()), C.byref(_mlp((64, 64), 1))))
    assert _policy(lib, stride=words + 2) == PDX_ERR_INVALID
    assert _policy(lib, stride=words - 4) == PDX_ERR_INVALID


def test_policy_step_members_rejects_plan_overflow(lib):
    # obs_dim 384 with 64-unit networks does not fit the policy kernel's shared-memory plan
    pi = _mlp((64, 64))
    stride = int(lib.pdx_policy_pack_words(384, C.byref(pi), C.byref(_mlp((64, 64), 1))))
    assert _policy(lib, obs_dim=384, pi=pi, stride=stride) == PDX_ERR_INVALID


# ---- pdx_gae_members / pdx_moments_members ----------------------------------------------------------
def _gae(lib, P=3, T=64, n=100, rew=FAKE, adv=FAKE):
    return lib.pdx_gae_members(P, T, n, rew, FAKE, FAKE, FAKE, FAKE, 0.99, 0.95, 1e-5, 1, FAKE, adv, FAKE, FAKE, None)


@pytest.mark.parametrize('case', [dict(P=0), dict(P=-2), dict(T=0), dict(n=0), dict(rew=None), dict(adv=None)])
def test_gae_members_rejects(lib, case):
    assert _gae(lib, **case) == PDX_ERR_INVALID


@pytest.mark.parametrize('case', [dict(P=0), dict(P=65536), dict(T=0), dict(n=0), dict(dim=0), dict(dim=1025),
                                  dict(x=None), dict(out=None)])
def test_moments_members_rejects(lib, case):
    a = dict(P=3, T=64, n=100, dim=34, x=FAKE, out=FAKE)
    a.update(case)
    assert lib.pdx_moments_members(a['P'], a['T'], a['n'], a['dim'], a['x'], None, a['out'], None) == PDX_ERR_INVALID


# ---- pdx_ppo_*_grad_members -------------------------------------------------------------------------
def _ppo_args(n=1000, obs_dim=34, hidden=(50, 50), n_out=4):
    b = L.PdxPpoBatch()
    b.n, b.obs_dim = n, obs_dim
    b.obs, b.act, b.adv, b.logp_old, b.target_v = FAKE, FAKE, FAKE, FAKE, FAKE
    g = L.PdxMlpGrad()
    for k in range(3):
        g.weight[k] = g.bias[k] = FAKE
    return b, _mlp(hidden, n_out), g


def _pi(lib, P=3, rows=1000, scratch=FAKE, scratch_bytes=BIG, **kw):
    b, m, g = _ppo_args(**kw)
    return lib.pdx_ppo_pi_grad_members(P, C.byref(b), rows, None, C.byref(m), FAKE, 0.2, C.byref(g), FAKE, None,
                                       None, None, scratch, scratch_bytes, None)


def _v(lib, P=3, rows=1000, scratch=FAKE, scratch_bytes=BIG, **kw):
    b, m, g = _ppo_args(n_out=1, **kw)
    return lib.pdx_ppo_v_grad_members(P, C.byref(b), rows, None, C.byref(m), C.byref(g), FAKE, scratch,
                                      scratch_bytes, None)


def _per_cta(obs_dim=34, hidden=(50, 50), n_out=4):
    h1, h2 = hidden
    return 8 * (h1 * (obs_dim + 1) + h2 * (h1 + 1) + n_out * (h2 + 1) + 2)


@pytest.mark.parametrize('fn', [_pi, _v])
@pytest.mark.parametrize('case', [
    dict(P=0), dict(P=-1), dict(P=65536), dict(n=0), dict(obs_dim=0), dict(obs_dim=385), dict(hidden=(65, 50)),
    dict(hidden=(50, 65)), dict(rows=999), dict(rows=0), dict(scratch=None),
])
def test_ppo_grad_members_rejects(lib, fn, case):
    assert fn(lib, **case) == PDX_ERR_INVALID


@pytest.mark.parametrize('fn,n_out', [(_pi, 4), (_v, 1)])
def test_ppo_grad_members_needs_one_cta_of_scratch_per_member(lib, fn, n_out):
    per = _per_cta(n_out=n_out)
    assert fn(lib, P=3, scratch_bytes=3 * per - 1) == PDX_ERR_INVALID
    assert fn(lib, P=1, scratch_bytes=per - 1) == PDX_ERR_INVALID


def test_ppo_grad_members_null_batch_pointers(lib):
    b, m, g = _ppo_args()
    b.act = None
    assert lib.pdx_ppo_pi_grad_members(3, C.byref(b), 1000, None, C.byref(m), FAKE, 0.2, C.byref(g), FAKE, None, None,
                                       None, FAKE, BIG, None) == PDX_ERR_INVALID
    b, m, g = _ppo_args(n_out=1)
    b.target_v = None
    assert lib.pdx_ppo_v_grad_members(3, C.byref(b), 1000, None, C.byref(m), C.byref(g), FAKE, FAKE, BIG,
                                      None) == PDX_ERR_INVALID
    b, m, g = _ppo_args()
    assert lib.pdx_ppo_pi_grad_members(3, C.byref(b), 1000, None, C.byref(m), None, 0.2, C.byref(g), FAKE, None, None,
                                       None, FAKE, BIG, None) == PDX_ERR_INVALID        # log_std
    assert lib.pdx_ppo_pi_grad_members(3, C.byref(b), 1000, None, C.byref(m), FAKE, -0.1, C.byref(g), FAKE, None,
                                       None, None, FAKE, BIG, None) == PDX_ERR_INVALID  # clip_ratio


@pytest.mark.parametrize('case', [dict(P=0), dict(numel=0), dict(param=None), dict(grad=None), dict(steps=None),
                                  dict(lr=-1.0), dict(beta1=1.0), dict(beta2=-0.1), dict(eps=-1.0)])
def test_adam_members_rejects(lib, case):
    a = dict(P=3, numel=100, param=FAKE, grad=FAKE, steps=FAKE, lr=3e-4, beta1=0.9, beta2=0.999, eps=1e-8)
    a.update(case)
    assert lib.pdx_adam_members(a['P'], a['numel'], a['param'], a['grad'], FAKE, FAKE, a['steps'], None, a['lr'],
                                a['beta1'], a['beta2'], a['eps'], None) == PDX_ERR_INVALID


# ---- PopulationPPO -----------------------------------------------------------------------------------
class _FakeDist:
    def __init__(self, world):
        self.world = world

    def is_initialized(self):
        return True

    def get_world_size(self):
        return self.world


def test_population_rejects_several_ranks():
    with pytest.raises(ValueError, match='one GPU'):
        PopulationPPO('DroneHoverSimpleEnv-v0', members=2, dist=_FakeDist(2))


@pytest.mark.parametrize('kernel', ['tc', 'Torch', None, 'triton'])
def test_population_rejects_bad_update_kernel(kernel):
    with pytest.raises(ValueError, match='update_kernel'):
        PopulationPPO('DroneHoverSimpleEnv-v0', members=2, update_kernel=kernel)


def test_population_rejects_float64_environments():
    # the member policy step and GAE read the rollout's observations and rewards as float32
    import torch
    with pytest.raises(ValueError, match='float32'):
        PopulationPPO('DroneHoverSimpleEnv-v0', members=2, dtype=torch.float64)
    with pytest.raises(ValueError, match='philox'):
        PopulationPPO('DroneHoverSimpleEnv-v0', members=2, rng='tape')


@pytest.mark.parametrize('kw', [dict(members=0), dict(num_envs_per_member=0), dict(device='cpu')])
def test_population_rejects_bad_shapes_and_devices(kw):
    with pytest.raises(ValueError):
        PopulationPPO('DroneHoverSimpleEnv-v0', **kw)
