"""NPG / TRPO populations without a GPU: pdx_ppo_pi_fvp_members' argument checks at the C ABI, the batched
conjugate-gradient solve and line search against their single-agent loops, and the constructor's rejections."""
import ctypes as C
import math
import os

import pytest
import torch

from phoenix_drone_simulation_b200 import lib as L
from phoenix_drone_simulation_b200.npg import conjugate_gradients
from phoenix_drone_simulation_b200.population import (PopulationNPG, PopulationTRPO, conjugate_gradients_members,
                                                      line_search_members)
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


def _count(obs_dim, hidden):
    h1, h2 = hidden
    return h1 * (obs_dim + 1) + h2 * (h1 + 1) + 4 * (h2 + 1)


def _place(st, obs_dim, hidden, base):
    """Points the six tensors of `st` back to back from `base` (member 0's row of a flat [P][F] vector)."""
    k = base
    for i, (r, c) in enumerate([(hidden[0], obs_dim), (hidden[1], hidden[0]), (4, hidden[1])]):
        st.weight[i] = k
        k += 4 * r * c
        st.bias[i] = k
        k += 4 * r
    return k


def _args(P=3, n=1000, obs_dim=34, hidden=(50, 50)):
    b = L.PdxPpoBatch()
    b.n, b.obs_dim, b.obs = n, obs_dim, FAKE
    pi = L.PdxMlp()
    pi.hidden[0], pi.hidden[1], pi.n_out = hidden[0], hidden[1], 4
    for k in range(3):
        pi.weight[k] = pi.bias[k] = FAKE
    d = L.PdxMlp()
    d.hidden[0], d.hidden[1], d.n_out = hidden[0], hidden[1], 4
    F = _count(obs_dim, hidden)
    _place(d, obs_dim, hidden, 0x100000)
    out = L.PdxMlpGrad()
    _place(out, obs_dim, hidden, 0x100000 + 4 * P * F)        # right after dir's [P][F]
    per_cta = 8 * (F + 2)
    return {'P': P, 'b': b, 'rows': n, 'active': None, 'pi': pi, 'log_std': FAKE, 'dir': d, 'scale': 0.25,
            'damping': 0.1, 'out': out, 'stride': F, 'scratch': FAKE, 'scratch_bytes': P * per_cta}


def _call(lib, a):
    r = lambda x: C.byref(x) if x is not None else None
    return lib.pdx_ppo_pi_fvp_members(a['P'], r(a['b']), a['rows'], a['active'], r(a['pi']), a['log_std'], r(a['dir']),
                                      a['scale'], a['damping'], r(a['out']), a['stride'], a['scratch'],
                                      a['scratch_bytes'], None)


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the behaviour WITHOUT a GPU')
def test_valid_calls_without_device_report_no_device(lib):
    for kw in ({}, {'P': 1, 'n': 1, 'obs_dim': 384, 'hidden': (64, 64)}, {'P': 7, 'obs_dim': 37, 'hidden': (7, 33)}):
        a = _args(**kw)
        assert _call(lib, a) == PDX_ERR_NO_DEVICE
        assert 'no CPU path' in lib.pdx_last_error().decode()
        a['b'].index, a['rows'], a['active'], a['scale'], a['damping'] = FAKE, 1, FAKE, -3.0, 0.0
        assert _call(lib, a) == PDX_ERR_NO_DEVICE
        a = _args(**kw)
        a['stride'] += 12                                     # padded rows: out starts after dir's padded extent
        _place(a['out'], a['b'].obs_dim, tuple(a['pi'].hidden), 0x100000 + 4 * a['P'] * a['stride'])
        assert _call(lib, a) == PDX_ERR_NO_DEVICE


BAD = ['no_batch', 'n_0', 'obs_dim_0', 'obs_dim_385', 'no_obs', 'no_pi', 'pi_hidden_65', 'pi_n_out', 'pi_no_weight',
       'no_log_std', 'no_dir', 'dir_hidden', 'dir_no_bias', 'no_out', 'out_no_weight', 'scale_nan', 'scale_inf',
       'damping_negative', 'damping_nan', 'members_0', 'members_negative', 'members_65536', 'rows_below_n',
       'rows_0_indexed', 'stride_below_F', 'stride_negative', 'no_scratch', 'scratch_one_member_short',
       'out_aliases_dir', 'out_inside_last_member_of_dir', 'dir_inside_last_member_of_out', 'interleaved_rows']


@pytest.mark.parametrize('name', BAD)
def test_fvp_members_bad_arguments_are_invalid(lib, name):
    a = _args()
    b, pi, d, out, P, F = a['b'], a['pi'], a['dir'], a['out'], a['P'], a['stride']
    if name == 'no_batch': a['b'] = None
    elif name == 'n_0': b.n = 0
    elif name == 'obs_dim_0': b.obs_dim = 0
    elif name == 'obs_dim_385': b.obs_dim = 385
    elif name == 'no_obs': b.obs = None
    elif name == 'no_pi': a['pi'] = None
    elif name == 'pi_hidden_65': pi.hidden[1] = d.hidden[1] = 65
    elif name == 'pi_n_out': pi.n_out = d.n_out = 1
    elif name == 'pi_no_weight': pi.weight[1] = None
    elif name == 'no_log_std': a['log_std'] = None
    elif name == 'no_dir': a['dir'] = None
    elif name == 'dir_hidden': d.hidden[0] = 49
    elif name == 'dir_no_bias': d.bias[1] = None
    elif name == 'no_out': a['out'] = None
    elif name == 'out_no_weight': out.weight[2] = None
    elif name == 'scale_nan': a['scale'] = math.nan
    elif name == 'scale_inf': a['scale'] = math.inf
    elif name == 'damping_negative': a['damping'] = -0.1
    elif name == 'damping_nan': a['damping'] = math.nan
    elif name == 'members_0': a['P'] = 0
    elif name == 'members_negative': a['P'] = -2
    elif name == 'members_65536': a['P'] = 65536
    elif name == 'rows_below_n': a['rows'] = b.n - 1
    elif name == 'rows_0_indexed': b.index, a['rows'] = FAKE, 0
    elif name == 'stride_below_F': a['stride'] = F - 1
    elif name == 'stride_negative': a['stride'] = -F
    elif name == 'no_scratch': a['scratch'] = None
    elif name == 'scratch_one_member_short': a['scratch_bytes'] -= 1
    elif name == 'out_aliases_dir': _place(out, 34, (50, 50), 0x100000)
    # member 0's out clears member 0's dir, but lies inside the last member's dir
    elif name == 'out_inside_last_member_of_dir': _place(out, 34, (50, 50), 0x100000 + 4 * (P - 1) * F)
    elif name == 'dir_inside_last_member_of_out':
        _place(out, 34, (50, 50), 0x100000)
        _place(d, 34, (50, 50), 0x100000 + 4 * (P - 1) * F + 8)
    elif name == 'interleaved_rows':                         # one [P][2F] buffer: dir at [:, :F], out at [:, F:]
        a['stride'] = 2 * F
        _place(out, 34, (50, 50), 0x100000 + 4 * F)
    assert _call(lib, a) == PDX_ERR_INVALID, name
    assert lib.pdx_last_error().decode()


# ---- the batched conjugate-gradient solve ------------------------------------------------------------------------------
def _spd(P, n, seed):
    g = torch.Generator().manual_seed(seed)
    A = []
    for _ in range(P):
        Q, _ = torch.linalg.qr(torch.randn(n, n, generator=g, dtype=torch.float64))
        A.append(Q @ torch.diag(torch.linspace(0.5, 60.0, n, dtype=torch.float64)) @ Q.T)
    return torch.stack(A), g


@pytest.mark.parametrize('nsteps', [1, 4, 10, 30])
def test_batched_cg_equals_the_single_loop_per_member(nsteps):
    P, n = 4, 12
    A, g = _spd(P, n, nsteps)
    b = torch.randn(P, n, generator=g, dtype=torch.float64)
    # member 1's right-hand side lies in one eigenspace: CG solves it in one product, its residual (eps / (lambda |b|)
    # ~ 2e-11 with the reference's eps = 1e-6) drops below the tolerance and it leaves the loop at once, exactly where
    # the single loop breaks
    w, V = torch.linalg.eigh(A[1])
    b[1] = 1e3 * V[:, -1]
    calls, actives = [], []

    def avp(p, active):
        calls.append(p.clone())
        actives.append(active.clone())
        z = torch.einsum('pij,pj->pi', A, p)
        return torch.where(active.unsqueeze(1), z, torch.full_like(z, math.nan))   # inactive rows: garbage
    x = conjugate_gradients_members(avp, b, nsteps)
    for m in range(P):
        count = []

        def one(v, m=m):
            count.append(1)
            return A[m] @ v
        ref = conjugate_gradients(one, b[m].clone(), nsteps)
        torch.testing.assert_close(x[m], ref, rtol=1e-10, atol=1e-13)   # row sums for torch.dot
        # member m took part in exactly the products the single loop made
        assert sum(bool(a[m]) for a in actives) == len(count), (m, len(count))
    if 1 < nsteps <= 10:
        assert actives[0].tolist() == [True] * P and actives[1].tolist() == [True, False, True, True]
        assert len(calls) == nsteps                           # the other members run every iteration
    w_ref = torch.linalg.solve(A[1], b[1])
    torch.testing.assert_close(x[1], w_ref, rtol=1e-9, atol=1e-12)


def test_batched_cg_stops_when_every_member_has_converged():
    P, n = 3, 6
    A, _ = _spd(P, n, 7)
    b = torch.stack([1e3 * torch.linalg.eigh(A[m])[1][:, -1 - m] for m in range(P)])
    calls = []
    conjugate_gradients_members(lambda p, active: calls.append(1) or torch.einsum('pij,pj->pi', A, p), b, 10)
    assert len(calls) == 1


# ---- the batched line search ------------------------------------------------------------------------------------------
def _objective(m):
    """Member m's (improvement, kl) at theta = theta_old + t: member 0 passes candidate 1; member 1 loses ground until
    2 |t|^2 <= 1 and passes candidate 3 (fraction 0.64); member 2 never improves and rejects all 15."""
    def f(t, step):
        if m == 0:
            return (t * step).sum(), 0.001 * (t * t).sum() / (step * step).sum()
        if m == 1:
            return (t * step).sum() * (1.0 - 2.0 * (t * t).sum()), 0.004 * (t * t).sum() / (step * step).sum()
        return -(t * t).sum() - 1e-3, 0.0 * (t * t).sum()
    return f


def test_batched_line_search_equals_the_single_search_per_member():
    g = torch.Generator().manual_seed(3)
    P, F, target_kl = 3, 9, 0.002
    theta_old = torch.randn(P, F, generator=g)
    step = torch.randn(P, F, generator=g)
    step[1] *= 1.1 / float(step[1].norm())
    fns = [_objective(m) for m in range(P)]

    def host(m, theta):
        """float32 device scalars read back as host floats, as NPG's evaluate does."""
        i, k = fns[m](theta - theta_old[m], step[m])
        return float(torch.stack([i, k])[0]), float(torch.stack([i, k])[1])
    tried = []

    def evaluate(theta, active):
        tried.append(active.tolist())
        vals = [host(m, theta[m]) for m in range(P)]
        return [v[0] for v in vals], [v[1] for v in vals]
    final, accept = line_search_members(evaluate, step, theta_old, target_kl)
    for m in range(P):
        ref_step, ref_accept = line_search(lambda theta, m=m: host(m, theta), step[m], theta_old[m], target_kl)
        assert accept[m] == ref_accept, (m, accept, ref_accept)
        assert torch.equal(final[m], ref_step), m
    assert accept == [1, 3, 0], accept
    assert len(tried) == 15
    assert tried[0] == [True] * P and tried[1] == [False, True, True] and tried[3] == [False, False, True]
    assert bool((final[2] == 0).all())


# ---- constructor -----------------------------------------------------------------------------------------------------
class _FakeDist:
    def is_initialized(self):
        return True

    def get_world_size(self):
        return 2


@pytest.mark.parametrize('cls', [PopulationNPG, PopulationTRPO])
@pytest.mark.parametrize('kw,match', [
    (dict(dist=_FakeDist()), 'one GPU'), (dict(device='cpu'), 'CUDA'), (dict(dtype=torch.float64), 'float32'),
    (dict(rng='tape'), 'philox'), (dict(update_kernel='triton'), 'update_kernel'), (dict(update_kernel=None), 'update_kernel'),
    (dict(members=0), 'members'),
])
def test_population_npg_trpo_inherit_the_rejections(cls, kw, match):
    kw = {'members': 2, **kw}
    with pytest.raises(ValueError, match=match):
        cls('DroneHoverSimpleEnv-v0', **kw)
