"""NPG / TRPO without a GPU: pdx_ppo_pi_fvp's argument checks at the C ABI, the conjugate-gradient loop, the torch
Fisher-vector product, the flat parameter order and TRPO's step-size decision."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.npg import KL_SCALE, conjugate_gradients
from phoenix_drone_simulation_b200.ppo import flat_views, pi_flat_params, pi_fvp_torch, pi_net_params
from phoenix_drone_simulation_b200.rollout import ActorCritic
from phoenix_drone_simulation_b200.trpo import line_search

PDX_ERR_INVALID, PDX_ERR_NO_DEVICE = -1, -3
FAKE = 0x1000          # never dereferenced: every check below happens before the library touches memory
BIG = 1 << 30


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(L.LIB_PATH):
        from phoenix_drone_simulation_b200.build import build
        build()
    return L.load()


def _mlp(hidden, n_out):
    m = L.PdxMlp()
    m.hidden[0], m.hidden[1], m.n_out = hidden[0], hidden[1], n_out
    return m


def _place(st, obs_dim, hidden, base):
    """Points the six tensors of `st` back to back from `base` (the layout of ppo.flat_views); returns the end."""
    sizes = [(hidden[0], obs_dim), (hidden[1], hidden[0]), (4, hidden[1])]
    k = base
    for i, (r, c) in enumerate(sizes):
        st.weight[i] = k
        k += 4 * r * c
        st.bias[i] = k
        k += 4 * r
    return k


def _fvp_args(n=1000, obs_dim=34, hidden=(50, 50)):
    b = L.PdxPpoBatch()
    b.n, b.obs_dim, b.obs = n, obs_dim, FAKE
    pi = _mlp(hidden, 4)
    for k in range(3):
        pi.weight[k] = pi.bias[k] = FAKE
    d = _mlp(hidden, 4)
    end = _place(d, obs_dim, hidden, 0x100000)
    out = L.PdxMlpGrad()
    _place(out, obs_dim, hidden, end)
    return {'b': b, 'pi': pi, 'log_std': FAKE, 'dir': d, 'scale': 0.25, 'damping': 0.1, 'out': out,
            'scratch': FAKE, 'scratch_bytes': BIG}


def _fvp(lib, a):
    r = lambda x: C.byref(x) if x is not None else None
    return lib.pdx_ppo_pi_fvp(r(a['b']), r(a['pi']), a['log_std'], r(a['dir']), a['scale'], a['damping'], r(a['out']),
                              a['scratch'], a['scratch_bytes'], None)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
def test_valid_calls_without_device_report_no_device(lib):
    for kw in ({}, {'n': 1, 'obs_dim': 384, 'hidden': (64, 64)}, {'obs_dim': 37, 'hidden': (7, 33)}):
        a = _fvp_args(**kw)
        assert _fvp(lib, a) == PDX_ERR_NO_DEVICE
        assert 'no CPU path' in lib.pdx_last_error().decode()
        a['b'].index, a['scale'], a['damping'] = FAKE, -3.0, 0.0      # any finite scale, damping 0
        assert _fvp(lib, a) == PDX_ERR_NO_DEVICE
    # the unclipped surrogate: clip_ratio = +inf is a valid call of pdx_ppo_pi_grad
    b = L.PdxPpoBatch()
    b.n, b.obs_dim = 1000, 34
    b.obs = b.act = b.adv = b.logp_old = FAKE
    m = _mlp((50, 50), 4)
    g = L.PdxMlpGrad()
    for k in range(3):
        m.weight[k] = m.bias[k] = g.weight[k] = g.bias[k] = FAKE
    for grad in (C.byref(g), None):
        assert lib.pdx_ppo_pi_grad(C.byref(b), C.byref(m), FAKE, math.inf, grad, FAKE, None, None, None, FAKE, BIG,
                                   None) == PDX_ERR_NO_DEVICE


BAD = ['no_batch', 'n_0', 'n_negative', 'obs_dim_0', 'obs_dim_385', 'no_obs', 'no_pi', 'pi_hidden_65', 'pi_hidden_0',
       'pi_n_out', 'pi_no_weight', 'pi_no_bias', 'no_log_std', 'no_dir', 'dir_hidden', 'dir_n_out', 'dir_no_weight',
       'dir_no_bias', 'no_out', 'out_no_weight', 'out_no_bias', 'out_aliases_dir', 'out_overlaps_dir', 'scale_nan',
       'scale_inf', 'damping_negative', 'damping_nan', 'damping_inf', 'no_scratch', 'scratch_small']


@pytest.mark.parametrize('name', BAD)
def test_fvp_bad_arguments_are_invalid(lib, name):
    a = _fvp_args()
    b, pi, d, out = a['b'], a['pi'], a['dir'], a['out']
    if name == 'no_batch': a['b'] = None
    elif name == 'n_0': b.n = 0
    elif name == 'n_negative': b.n = -5
    elif name == 'obs_dim_0': b.obs_dim = 0
    elif name == 'obs_dim_385': b.obs_dim = 385
    elif name == 'no_obs': b.obs = None
    elif name == 'no_pi': a['pi'] = None
    elif name == 'pi_hidden_65': pi.hidden[1] = d.hidden[1] = 65
    elif name == 'pi_hidden_0': pi.hidden[0] = d.hidden[0] = 0
    elif name == 'pi_n_out': pi.n_out = d.n_out = 1
    elif name == 'pi_no_weight': pi.weight[1] = None
    elif name == 'pi_no_bias': pi.bias[2] = None
    elif name == 'no_log_std': a['log_std'] = None
    elif name == 'no_dir': a['dir'] = None
    elif name == 'dir_hidden': d.hidden[0] = 49
    elif name == 'dir_n_out': d.n_out = 3
    elif name == 'dir_no_weight': d.weight[0] = None
    elif name == 'dir_no_bias': d.bias[1] = None
    elif name == 'no_out': a['out'] = None
    elif name == 'out_no_weight': out.weight[2] = None
    elif name == 'out_no_bias': out.bias[0] = None
    elif name == 'out_aliases_dir': _place(out, 34, (50, 50), 0x100000)
    elif name == 'out_overlaps_dir': out.bias[2] = d.weight[2] + 8
    elif name == 'scale_nan': a['scale'] = math.nan
    elif name == 'scale_inf': a['scale'] = math.inf
    elif name == 'damping_negative': a['damping'] = -0.1
    elif name == 'damping_nan': a['damping'] = math.nan
    elif name == 'damping_inf': a['damping'] = math.inf
    elif name == 'no_scratch': a['scratch'] = None
    elif name == 'scratch_small': a['scratch_bytes'] = 64
    assert _fvp(lib, a) == PDX_ERR_INVALID, name
    assert lib.pdx_last_error().decode()


@pytest.mark.parametrize('clip', [math.nan, -0.1, -math.inf])
def test_unclipped_surrogate_keeps_rejecting_nan_and_negative_clip(lib, clip):
    b = L.PdxPpoBatch()
    b.n, b.obs_dim = 1000, 34
    b.obs = b.act = b.adv = b.logp_old = FAKE
    m = _mlp((50, 50), 4)
    for k in range(3):
        m.weight[k] = m.bias[k] = FAKE
    assert lib.pdx_ppo_pi_grad(C.byref(b), C.byref(m), FAKE, clip, None, FAKE, None, None, None, FAKE, BIG,
                               None) == PDX_ERR_INVALID


def _reference_cg(Avp, b, nsteps, residual_tol=1e-10, eps=1e-6):
    """algs/utils.py conjugate_gradients, literally (including the first product Avp(0))."""
    x = torch.zeros_like(b)
    r = b - Avp(x)
    p = r.clone()
    rdotr = torch.dot(r, r)
    iterates = []
    for i in range(nsteps):
        z = Avp(p)
        alpha = rdotr / (torch.dot(p, z) + eps)
        x += alpha * p
        r -= alpha * z
        iterates.append(x.clone())
        new_rdotr = torch.dot(r, r)
        if torch.sqrt(new_rdotr) < residual_tol:
            break
        mu = new_rdotr / (rdotr + eps)
        p = r + mu * p
        rdotr = new_rdotr
    return x, iterates


@pytest.mark.parametrize('nsteps', [1, 3, 10, 40])
def test_conjugate_gradients_match_the_reference_loop(nsteps):
    g = torch.Generator().manual_seed(nsteps)
    M = torch.randn(12, 12, generator=g, dtype=torch.float64)
    A = M @ M.T + 0.5 * torch.eye(12, dtype=torch.float64)
    b = torch.randn(12, generator=g, dtype=torch.float64)
    ref, iterates = _reference_cg(lambda v: A @ v, b, nsteps)
    for k, it in enumerate(iterates):                        # every iterate, by stopping after k + 1 products
        assert torch.equal(conjugate_gradients(lambda v: A @ v, b, k + 1), it)
    assert torch.equal(conjugate_gradients(lambda v: A @ v, b, nsteps), ref)
    if nsteps == 40:
        sol = np.linalg.solve(A.numpy(), b.numpy())
        # the eps terms of the reference bias the result slightly: it approaches the solve, it does not reach it
        assert np.abs(ref.numpy() - sol).max() <= 1e-4 * np.abs(sol).max()


def test_flat_order_is_the_reference_order():
    torch.manual_seed(0)
    ac = ActorCritic(34, device='cpu')
    ref = torch.cat([p.view(-1) for p in ac.pi.net.parameters()])
    assert torch.equal(pi_flat_params(ac), ref)
    assert all(p_ is not ac.log_std for p_ in pi_net_params(ac))
    for v, p_ in zip(flat_views(ref, pi_net_params(ac)), pi_net_params(ac)):
        assert torch.equal(v, p_) and v.data_ptr() >= ref.data_ptr()


@pytest.mark.parametrize('hidden,index', [((50, 50), False), ((7, 33), True)])
def test_torch_fvp_is_the_gauss_newton_product(hidden, index):
    """pi_fvp_torch (the reference's double backward) == J^T J v / (4 sigma^2) + damping v in float64."""
    torch.manual_seed(1)
    ac = ActorCritic(9, pi_hidden=hidden, device='cpu').double()
    ac.set_log_std(0.6)
    obs = torch.randn(40, 9, dtype=torch.float64)
    idx = torch.arange(0, 40, 4) if index else None
    params = pi_net_params(ac)
    theta = pi_flat_params(ac)
    v = torch.randn(theta.numel(), dtype=torch.float64)
    o = obs if idx is None else obs[idx]

    def mu_of(flat):
        ws = flat_views(flat, params)
        h = torch.relu(o @ ws[0].T + ws[1])
        h = torch.relu(h @ ws[2].T + ws[3])
        return (h @ ws[4].T + ws[5]).reshape(-1)

    J = torch.autograd.functional.jacobian(mu_of, theta)        # [rows * 4, P]
    var = torch.exp(2 * ac.log_std).repeat(o.shape[0])
    expect = J.T @ (J @ v / var) / (4 * o.shape[0]) + 0.1 * v
    got = pi_fvp_torch(ac, obs, v, 0.1, KL_SCALE, index=idx)
    torch.testing.assert_close(got, expect, rtol=1e-10, atol=1e-12)
    got1 = pi_fvp_torch(ac, obs, v, 0.0, 1.0, index=idx)        # scale 1: the summed KL's Hessian
    torch.testing.assert_close(got1, 4 * (expect - 0.1 * v), rtol=1e-10, atol=1e-12)


def _search(table, target_kl=0.01):
    """line_search over candidates j whose (improvement, kl) come from table[j]; returns (frac, accept, tried)."""
    tried = []

    def evaluate(theta):
        j = len(tried)
        tried.append(float(theta[0]))
        return table[j] if j < len(table) else (-1.0, 0.0)
    step, accept = line_search(evaluate, torch.tensor([1.0]), torch.tensor([0.0]), target_kl)
    return float(step[0]), accept, tried


def test_line_search_accepts_the_first_candidate_that_passes():
    frac, accept, tried = _search([(-1e-3, 0.001), (1e-3, 0.02), (0.0, 0.015)])
    assert accept == 3 and frac == pytest.approx(0.64) and tried == pytest.approx([1.0, 0.8, 0.64])


@pytest.mark.parametrize('bad', [(math.nan, 0.001), (math.inf, 0.001), (-math.inf, 0.001), (-1e-6, 0.001),
                                 (1.0, 0.0150001), (1.0, math.nan)])
def test_line_search_rejects(bad):
    frac, accept, tried = _search([bad, (0.5, 0.001)])
    assert accept == 2 and frac == pytest.approx(0.8)


def test_line_search_returns_a_zero_step_when_nothing_passes():
    frac, accept, tried = _search([(-1.0, 0.0)] * 15)
    assert accept == 0 and frac == 0.0 and len(tried) == 15
    assert tried[-1] == pytest.approx(0.8 ** 14)
