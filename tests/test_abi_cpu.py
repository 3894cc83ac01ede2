"""CPU-side checks of the drop-in boundary: the C-ABI library loads, exports every symbol
that include/phoenix_b200.h declares, its structs match the ctypes mirror, the query
functions agree with the golden fixtures, and -- with no CUDA device -- every compute entry
point FAILS LOUDLY (there is no CPU fallback on the product path)."""
import ctypes as C
import os
import re

import numpy as np
import pytest
import torch

import phoenix_drone_simulation_b200 as pds
from phoenix_drone_simulation_b200 import lib as L
from golden_util import golden_names, load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(L.LIB_PATH):
        from phoenix_drone_simulation_b200.build import build
        build()
    return L.load()


def test_header_symbols_are_exported(lib):
    header = open(os.path.join(ROOT, 'include', 'phoenix_b200.h')).read()
    header = re.sub(r'/\*.*?\*/', '', header, flags=re.S)
    declared = set(re.findall(r'\b(pdx_[a-z_0-9]+)\s*\(', header))
    assert declared == set(L.EXPORTED_SYMBOLS)
    for name in declared:
        assert hasattr(lib, name), name


def test_struct_sizes_and_version(lib):
    assert lib.pdx_abi_version() == L.ABI_VERSION
    assert lib.pdx_config_size() == C.sizeof(L.PdxConfig)
    assert lib.pdx_buffers_size() == C.sizeof(L.PdxBuffers)


@pytest.mark.parametrize('env_id,obs_dim', [
    ('DroneHoverSimpleEnv-v0', 34), ('DroneHoverBulletEnv-v0', 34), ('DroneCircleSimpleEnv-v0', 40),
    ('DroneCircleBulletEnv-v0', 40), ('DroneTakeOffSimpleEnv-v0', 48), ('DroneTakeOffBulletEnv-v0', 48)])
def test_observation_widths(lib, env_id, obs_dim):
    """D = H (C + 4): 34 / 40 / 48 at H = 2 (SURVEY 8; verified by running the reference)."""
    c = pds.EnvConfig(env_id).to_pdx()
    assert c.obs_dim == obs_dim
    c = pds.EnvConfig(env_id, observation_history_size=8).to_pdx()
    assert c.obs_dim == 4 * obs_dim


def test_noise_off_hover_width(lib):
    assert pds.EnvConfig('DroneHoverSimpleEnv-v0', observation_noise=0).to_pdx().obs_dim == 42


@pytest.mark.parametrize('name', golden_names())
def test_tape_slots_match_reference_draw_counts(lib, name):
    """The per-phase draw counts of the engine equal what the unmodified reference consumed."""
    g = load_golden(name)
    kw = dict(g['kwargs'])
    c = pds.EnvConfig(g['env_id'], **kw).to_pdx()
    rs, ss, is_ = C.c_int(), C.c_int(), C.c_int()
    assert lib.pdx_tape_slots(C.byref(c), C.byref(rs), C.byref(ss), C.byref(is_)) == 0
    assert ss.value == g['step_tape'].shape[1]
    assert rs.value == g['reset_tape'].shape[1]
    assert is_.value == g['init_tape'].shape[0]
    assert c.obs_dim == g['obs'].shape[1]


def test_state_layout(lib):
    c = pds.EnvConfig('DroneHoverSimpleEnv-v0').to_pdx()
    fw, nw = C.c_int(), C.c_int()
    seen = set()
    for name in ('xyz', 'vel', 'rpy', 'omega', 'ou', 'last_action', 'ep_return', 'ep_length',
                 'gyro_bias', 'gyro_lpf', 'dt', 'mass', 'inertia', 'ftf1'):
        assert lib.pdx_state_field(C.byref(c), name.encode(), C.byref(fw), C.byref(nw)) == 0
        words = set(range(fw.value, fw.value + nw.value))
        assert not (words & seen), name
        seen |= words
    assert len(seen) == 34                      # 28 per-step words + 6 per-episode constants
    # bookkeeping word of the reset-package pool (4 * auto-resets consumed + pending-slot bits)
    assert lib.pdx_state_field(C.byref(c), b'ep_index', C.byref(fw), C.byref(nw)) == 0 and nw.value == 1
    assert fw.value not in seen
    assert lib.pdx_state_field(C.byref(c), b'hist', C.byref(fw), C.byref(nw)) == 0
    assert fw.value == 36 and nw.value == 20    # one history slot: 13 + 4 words in 5 quads
    assert lib.pdx_state_field(C.byref(c), b'pool', C.byref(fw), C.byref(nw)) == 0
    assert fw.value == 56 and nw.value == 4 * 16 * 4    # four reset packages: 9 state quads + 26 observation words each
    assert lib.pdx_state_quads(C.byref(c)) == 14 + 64
    assert lib.pdx_state_field(C.byref(c), b'quat', C.byref(fw), C.byref(nw)) != 0     # Bullet only
    assert b'does not exist' in lib.pdx_last_error()
    # algorithmic bytes per env (DESIGN.md): state 34 + history 17 words read and written once
    # per launch; per step obs 34 + reward + cost words, 16 B action, 2 flag bytes
    assert lib.pdx_step_bytes(C.byref(c)) == (51 + 51 + 34 + 2) * 4 + 16 + 2
    lib.pdx_rollout_bytes.restype = C.c_int64
    assert lib.pdx_rollout_bytes(C.byref(c), 64) == (51 + 51) * 4 + 64 * ((34 + 2) * 4 + 16 + 2)


def test_pid_control_modes_add_twelve_state_words(lib):
    """AttitudeRate / Attitude (envs/control.py:120-287): integrals and last errors of both loops."""
    fw, nw = C.c_int(), C.c_int()
    base = pds.EnvConfig('DroneHoverBulletEnv-v0').to_pdx()
    assert lib.pdx_state_field(C.byref(base), b'pid', C.byref(fw), C.byref(nw)) != 0
    for mode, code in (('AttitudeRate', 1), ('Attitude', 2)):
        c = pds.EnvConfig('DroneHoverBulletEnv-v0', control_mode=mode, aggregate_phy_steps=4).to_pdx()
        assert c.control_mode == code and c.agg == 4
        assert lib.pdx_state_field(C.byref(c), b'pid', C.byref(fw), C.byref(nw)) == 0 and nw.value == 12
        assert lib.pdx_state_quads(C.byref(c)) >= lib.pdx_state_quads(C.byref(base)) + 3 - 1
        assert c.obs_dim == base.obs_dim


def test_unsupported_configurations_are_rejected(lib):
    with pytest.raises(NotImplementedError):
        pds.EnvConfig('DroneHoverSimpleEnv-v0', control_mode='Position')
    with pytest.raises(KeyError):
        pds.EnvConfig('DroneFooEnv-v0')
    with pytest.raises(L.PhoenixB200Error):
        pds.EnvConfig('DroneHoverBulletEnv-v0', aggregate_phy_steps=1).to_pdx()   # agg % obs_rate
    with pytest.raises(L.PhoenixB200Error):
        pds.EnvConfig('DroneHoverSimpleEnv-v0', observation_history_size=0).to_pdx()


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
def test_no_cpu_fallback(lib):
    """Without a CUDA device the product path must raise, not silently compute on the CPU."""
    with pytest.raises(L.PhoenixB200Error):
        pds.VecEnv('DroneHoverSimpleEnv-v0', 4)
    with pytest.raises(L.PhoenixB200Error):
        pds.make('DroneHoverSimpleEnv-v0')
    c = pds.EnvConfig('DroneHoverSimpleEnv-v0').to_pdx()
    host = np.zeros(4096, dtype=np.float32)
    b = L.PdxBuffers()
    b.n_envs = 4
    for f in ('state', 'obs', 'reward', 'cost', 'terminated', 'truncated'):
        setattr(b, f, host.ctypes.data)
    assert lib.pdx_step(C.byref(c), C.byref(b), host.ctypes.data, 0, 1, None) == -3     # PDX_ERR_NO_DEVICE
    assert b'no CPU path' in lib.pdx_last_error()
    assert lib.pdx_gae(4, 4, *([host.ctypes.data] * 5), 0.99, 0.95, 1.0, 0, None, *([host.ctypes.data] * 3), None) == -3


COMPUTE_ENTRY_POINTS = ['pdx_init', 'pdx_reset', 'pdx_step', 'pdx_step_many', 'pdx_gae', 'pdx_moments', 'pdx_oms_update',
                        'pdx_stats_combine', 'pdx_policy_pack', 'pdx_policy_step', 'pdx_policy_tc_pack', 'pdx_policy_step_tc',
                        'pdx_collect', 'pdx_evaluate']


def _mlp(h1, h2, n_out):
    m = L.PdxMlp()
    m.hidden[0], m.hidden[1], m.n_out = h1, h2, n_out
    return m


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
@pytest.mark.parametrize('entry', COMPUTE_ENTRY_POINTS)
def test_every_compute_entry_point_reports_no_device(lib, entry):
    """With arguments that pass validation and no CUDA device, every compute entry point returns PDX_ERR_NO_DEVICE
    and says there is no CPU path.  The pointers are never dereferenced: the device check comes first."""
    F = 0x1000
    c = pds.EnvConfig('DroneHoverSimpleEnv-v0').to_pdx()
    D = c.obs_dim
    b = L.PdxBuffers()
    b.n_envs = 4
    for f in ('state', 'obs', 'reward', 'cost', 'terminated', 'truncated'):
        setattr(b, f, F)
    pi, v = _mlp(50, 50, 4), _mlp(64, 64, 1)
    pol = L.PdxPolicy()
    pol.obs_dim, pol.precision, pol.pi, pol.v, pol.log_std, pol.packed = D, 1, C.pointer(pi), C.pointer(v), F, F
    ro = L.PdxRollout()
    ro.n_steps, ro.scratch_bytes = 8, 1 << 40
    for f in ('obs0', 'act', 'val', 'logp', 'last_val', 'scratch'):
        setattr(ro, f, F)
    ps = L.PdxPolicySet()
    ps.n_policies, ps.episodes, ps.obs_dim, ps.n_out, ps.stride, ps.packed = 2, 4, D, 4, 32 * 1024, F
    ps.hidden[0], ps.hidden[1] = 50, 50
    ev = L.PdxEvaluation()
    ev.ret, ev.cost, ev.length = F, F, F
    cfg, buf, pi_, v_ = C.byref(c), C.byref(b), C.byref(pi), C.byref(v)
    calls = {
        'pdx_init': lambda: lib.pdx_init(cfg, buf, 0, 1, None),
        'pdx_reset': lambda: lib.pdx_reset(cfg, buf, None, 0, 1, None),
        'pdx_step': lambda: lib.pdx_step(cfg, buf, F, 0, 1, None),
        'pdx_step_many': lambda: lib.pdx_step_many(cfg, buf, F, 8, 0, 1, None),
        'pdx_gae': lambda: lib.pdx_gae(8, 4, F, F, F, F, F, 0.99, 0.95, 1.0, 0, None, F, F, F, None),
        'pdx_moments': lambda: lib.pdx_moments(4, D, F, None, F, None),
        'pdx_oms_update': lambda: lib.pdx_oms_update(D, F, F, 4.0, 1, None, F, F, F, F, F, 3, None),
        'pdx_stats_combine': lambda: lib.pdx_stats_combine(1, F, F, None),
        'pdx_policy_pack': lambda: lib.pdx_policy_pack(D, pi_, v_, F, None),
        'pdx_policy_step': lambda: lib.pdx_policy_step(4, D, F, None, None, 0.0, pi_, v_, F, F, 0, 1, 0, F, F, F, None, None),
        'pdx_policy_tc_pack': lambda: lib.pdx_policy_tc_pack(D, pi_, v_, 1, F, None),
        'pdx_policy_step_tc': lambda: lib.pdx_policy_step_tc(4, D, F, None, None, 0.0, pi_, v_, F, F, 1, 0, 1, 0, F, F, F, None,
                                                             None),
        'pdx_collect': lambda: lib.pdx_collect(cfg, buf, C.byref(pol), C.byref(ro), 0, 1, None),
        'pdx_evaluate': lambda: lib.pdx_evaluate(cfg, buf, C.byref(ps), C.byref(ev), 0, 1, None),
    }
    assert sorted(calls) == sorted(COMPUTE_ENTRY_POINTS)
    assert lib.pdx_step(cfg, C.byref(L.PdxBuffers()), None, 0, 0, None) == -1   # a message that is not the one expected
    assert calls[entry]() == -3                                 # PDX_ERR_NO_DEVICE
    assert b'no CPU path' in lib.pdx_last_error()


def test_product_package_does_not_import_oracle():
    """The oracle is test infrastructure: nothing under the product package may reference it."""
    pkg = os.path.join(ROOT, 'phoenix_drone_simulation_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f


def test_empty_batch_is_rejected_before_any_cuda_call(lib):
    """n_envs = 0 (the 'empty input' edge case) is an argument error, reported without a device."""
    c = pds.EnvConfig('DroneHoverSimpleEnv-v0').to_pdx()
    b = L.PdxBuffers()
    b.n_envs = 0
    assert lib.pdx_step(C.byref(c), C.byref(b), None, 0, 0, None) == -1
    assert b'n_envs' in lib.pdx_last_error()
    assert lib.pdx_step_many(C.byref(c), C.byref(b), None, 0, 0, 0, None) == -1
    b.n_envs = 1 << 31                                   # the maximum shard: index products are 32 x 32 -> 64 bit
    assert lib.pdx_step(C.byref(c), C.byref(b), None, 0, 0, None) == -1
    assert b'2^31' in lib.pdx_last_error()


def test_tensor_core_policy_shape_checks_need_no_device(lib):
    """pdx_policy_tc_pack_words is pure host arithmetic: it sizes the packed image for shapes inside the
    tensor-core plan and rejects the others (callers then use pdx_policy_step)."""
    def mlp(h1, h2, n_out):
        m = L.PdxMlp()
        m.hidden[0], m.hidden[1], m.n_out = h1, h2, n_out
        return m
    pi, v = mlp(50, 50, 4), mlp(64, 64, 1)
    k1 = 40                                            # obs_dim 34 + the constant-1 column, padded to a multiple of 8
    b_words = k1 * 128 + 2 * 64 * 64 + 8 * 64 + 8 * (128 + 64 + 64)      # B1, B2a, B2c, collector bias tile, bias tiles
    assert lib.pdx_policy_tc_pack_words(34, C.byref(pi), C.byref(v), 1) == 336 + b_words
    assert lib.pdx_policy_tc_pack_words(34, C.byref(pi), C.byref(v), 3) == 336 + 2 * b_words
    assert lib.pdx_policy_tc_pack_words(34, C.byref(pi), C.byref(v), 2) == -1          # precision is 1 or 3
    assert lib.pdx_policy_tc_pack_words(160, C.byref(pi), C.byref(v), 3) == -1         # too wide
    assert lib.pdx_policy_tc_pack_words(40, C.byref(pi), C.byref(v), 1) == 336 + b_words + 8 * 128    # 40 -> K = 48
    assert lib.pdx_policy_tc_pack_words(48, C.byref(pi), C.byref(v), 1) == 336 + b_words + 8 * 128    # 48 -> K = 48
    assert lib.pdx_policy_tc_pack_words(34, C.byref(mlp(65, 50, 4)), C.byref(v), 3) == -1
    assert lib.pdx_policy_tc_pack_words(34, C.byref(pi), C.byref(mlp(64, 64, 2)), 3) == -1
    assert lib.pdx_policy_step_tc(0, 34, None, None, None, 0.0, C.byref(pi), C.byref(v), None, None, 3, 0, 0, 0,
                                  None, None, None, None, None) == -1
    # the fused collector validates its arguments before it touches the device
    c = pds.EnvConfig('DroneTakeOffSimpleEnv-v0').to_pdx()
    pol, out, b = L.PdxPolicy(), L.PdxRollout(), L.PdxBuffers()
    assert lib.pdx_collect(C.byref(c), C.byref(b), C.byref(pol), C.byref(out), 0, 0, None) == -1      # take-off rows are 48 wide
    assert b'pdx_collect' in lib.pdx_last_error()
    lib.pdx_collect_scratch_bytes.restype = C.c_int64
    assert lib.pdx_collect_scratch_bytes(0) >= 148 * 512 * 48


def test_flag_constants_match_the_header():
    """lib.py mirrors the #define'd flag bits of include/phoenix_b200.h (and the struct field they live in)."""
    import re
    header = open(os.path.join(ROOT, 'include', 'phoenix_b200.h')).read()
    defs = {m.group(1): int(m.group(2), 0) for m in re.finditer(r'#define\s+(PDX_[A-Z_]+)\s+(0x[0-9a-fA-F]+|\d+)\s*$', header, re.M)}
    assert defs['PDX_BUF_STATE_STABLE'] == L.PDX_BUF_STATE_STABLE
    assert defs['PDX_POLICY_TC_OVERLAP'] == L.PDX_POLICY_TC_OVERLAP
    assert 'flags' in [f[0] for f in L.PdxBuffers._fields_] and 'int32_t flags;' in header
    assert L.PDX_POLICY_TC_OVERLAP & 3 == 0          # must not collide with the precision values 1 and 3


def test_ids_are_registered_on_import():
    """phoenix_drone_simulation/__init__.py:8-50: importing the package registers the six ids with gymnasium when it
    is installed; the local make() is the registry otherwise."""
    import phoenix_drone_simulation_b200 as pds
    from phoenix_drone_simulation_b200 import envs
    assert set(envs.registry) == set(pds.ENV_IDS)
    try:
        import gymnasium
    except ImportError:
        assert envs.register_with_gymnasium() is False
        return
    for env_id in pds.ENV_IDS:
        assert env_id in gymnasium.envs.registry
