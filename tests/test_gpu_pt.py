"""Parallel tempering on the device (qb_pt_run, quinn_b200/csrc/qb_pt.cuh): bit identity with HMC / MALA at one
temperature on every gradient path, replay of the numpy oracle (tests/pt_oracle.py), determinism across call splits and
resumes, the tempered Gaussian posterior of a linear model, mode switching on a symmetric posterior, and the solver."""
import numpy as np
import pytest
import torch

import pt_oracle
from golden_util import netdesc_from_layers
from oracle import quinn_oracle as qo

pytestmark = pytest.mark.gpu


def _problem(layers, P, N, dtype, seed, in_dim, sigma=0.1):
    from quinn_b200 import ops
    rs = np.random.RandomState(seed)
    x = rs.rand(N, in_dim) * 2 - 1
    y = np.sin(2 * x.sum(1, keepdims=True)) + 0.1 * rs.randn(N, 1)
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, sigma, dtype=dtype, device='cuda')
    return prob, x, y, rs


PATHS = [  # name, layers, in_dim, dtype, plan code, tolerance, epsilon
    ('cuda_f64', qo.mlp_layers(1, 1, (5, 4), True, 'tanh'), 1, torch.float64, 0, 1e-9, 1e-2),
    ('stream_f64', qo.mlp_layers(10, 1, (128, 128, 128), True, 'tanh'), 10, torch.float64, 5, 1e-9, 2e-3),
    ('tcg_h32', qo.mlp_layers(2, 1, (32, 32), True, 'relu'), 2, torch.float32, 3, 2e-3, 1e-2),      # tanh ones go to TG8
    ('tg8_h64', qo.mlp_layers(3, 1, (64, 64), True, 'tanh'), 3, torch.float32, 4, 2e-3, 2e-3),
    ('tg8_h128', qo.mlp_layers(10, 1, (128, 128), True, 'tanh'), 10, torch.float32, 4, 2e-3, 2e-3),
    ('cuda_f32', qo.mlp_layers(1, 1, (5, 4), True, 'tanh'), 1, torch.float32, 0, 2e-3, 1e-2),
]


def _path(name):
    return [p for p in PATHS if p[0] == name][0]


def _start(prob, rs, K, P, dtype, scale=0.3):
    th = scale * rs.randn(K, P)
    return th.astype(np.float32).astype(np.float64) if dtype == torch.float32 else th


def _pt(prob, th0, betas, eps, nsteps, seed, G, method='hmc', L=3, swap_every=1, splits=(), store_every=1, chain_offset=0):
    """PT on the device over calls split at `splits`; th0 [G, P] starts every slot of its group"""
    from quinn_b200 import ops
    T = len(betas)
    st = ops.ChainState(prob, np.tile(th0, (T, 1)))
    ps = ops.PtState(st, G, betas, eps, L, method, swap_every)
    bounds = [0] + list(splits) + [nsteps]
    recs = []
    for a, b in zip(bounds[:-1], bounds[1:]):
        rec = ops.Recorder(st, b - a, store_every=store_every, sample_rows=G)
        ops.pt_run(st, ps, b - a, rec, seed=seed, chain_offset=chain_offset)
        recs.append(rec)
    torch.cuda.synchronize()
    return st, ps, recs


def _cat(recs, key):
    return torch.cat([getattr(r, key) for r in recs if getattr(r, key) is not None], 1).cpu().numpy()


def _snapshot(st, ps, recs):
    out = dict(theta=st.theta, lp=st.lp, map_theta=st.map_theta, map_lp=st.map_lp, naccept=st.naccept,
               grad_cur=ps.grad_cur, replica=ps.replica, last_end=ps.last_end, round_trips=ps.round_trips,
               swap_attempts=ps.swap_attempts, swap_accepts=ps.swap_accepts)
    out = {k: v.cpu().numpy() for k, v in out.items()}
    for key in ('logpost', 'alpha', 'accepted', 'samples'):
        out[key] = _cat(recs, key)
    out['logpost0'] = recs[0].logpost0.cpu().numpy()
    return out


# ---------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize('method', ['hmc', 'mala'])
@pytest.mark.parametrize('name', [p[0] for p in PATHS])
def test_one_temperature_is_bit_identical_to_hmc(name, method):
    """T = 1: the wrapper multiplies by exactly 1.0, so every record, state and MAP equals qb_hmc_run's bit for bit"""
    from quinn_b200 import ops
    _, (layers, P), in_dim, dtype, code, _, eps = _path(name)
    K, nsteps = 16, 6
    prob, x, y, rs = _problem(layers, P, 64, dtype, 5, in_dim)
    assert prob.plan_info(K, True)['tensor_core'] == code
    th0 = _start(prob, rs, K, P, dtype)
    st = ops.ChainState(prob, th0)
    hm = ops.HmcState(st, epsilon=eps, L=3, method=method)
    rec = ops.Recorder(st, nsteps, store_every=1)
    ops.hmc_run(st, hm, nsteps, rec, seed=21, chain_offset=3)
    st2, ps, recs = _pt(prob, th0, [1.0], eps, nsteps, 21, K, method=method, chain_offset=3)
    ref = dict(theta=st.theta, lp=st.lp, map_theta=st.map_theta, map_lp=st.map_lp, naccept=st.naccept,
               grad_cur=hm.grad_cur, logpost=rec.logpost, alpha=rec.alpha, accepted=rec.accepted, samples=rec.samples,
               logpost0=rec.logpost0)
    got = _snapshot(st2, ps, recs)
    for k, v in ref.items():
        v = v.cpu().numpy()
        assert v.tobytes() == got[k].tobytes(), (name, method, k)


# ---------------------------------------------------------------------------------------------------------------- 2
def _oracle(layers, x, y, sigma, th0, nsteps, betas, eps, method=0, swap_every=1, seed=0, chain_offset=0):
    lpg = lambda th: qo.logpost_grad(layers, th, x, y, sigma)           # noqa: E731
    return pt_oracle.run(lpg, th0, nsteps, betas, eps, method=method, L=3, swap_every=swap_every, seed=seed,
                         chain_offset=chain_offset)


def _first_close_call(orec, nsteps, swap_every, tol):
    """the first step whose MH decision, or the swap round after it, had a margin <= tol (nsteps if none)"""
    for s in range(nsteps):
        if orec['mh_margin'][:, s].min() <= tol:
            return s
        if (s + 1) % swap_every == 0 and min(m for *_, m in orec['swaps'][(s + 1) // swap_every - 1]) <= tol:
            return s
    return nsteps


def _compare(dev, ost, orec, G, nsteps, swap_every, tol, chain_offset=0):
    s_ok = _first_close_call(orec, nsteps, swap_every, tol)
    assert s_ok >= nsteps // 2, s_ok
    lp = orec['lp'][:, :s_ok]
    assert np.abs(dev['logpost'][:, :s_ok] - lp).max() <= tol * np.abs(lp).max()
    cz = orec['cold_z'][:s_ok].transpose(1, 0, 2)                      # [G, s, P]
    assert np.abs(dev['samples'][:, :s_ok] - cz).max() <= tol * max(np.abs(cz).max(), 1.0)
    np.testing.assert_array_equal(dev['accepted'][:, :s_ok].astype(bool), orec['acc'][:, :s_ok])
    if s_ok == nsteps:
        for key, okey in (('replica', 'replica'), ('swap_attempts', 'attempts'), ('swap_accepts', 'accepts'),
                          ('round_trips', 'round_trips'), ('naccept', 'naccept')):
            np.testing.assert_array_equal(dev[key], ost[okey], err_msg=key)
        assert np.abs(dev['theta'] - ost['z']).max() <= tol * max(np.abs(ost['z']).max(), 1.0)
        np.testing.assert_allclose(dev['map_lp'], ost['map_lp'], rtol=tol)
    return s_ok


NETS = {
    'mlp': (qo.mlp_layers(1, 1, (5, 4), True, 'tanh'), 1),
    'rnet_c1': (qo.rnet_layers(3, 3, 1, 1, biasorno=True, nonlin=True, mlp=False, shared=True), 1),
}
BETAS4 = [1.0, 0.6, 0.35, 0.2]


@pytest.mark.parametrize('swap_every', [1, 3])
@pytest.mark.parametrize('name', ['mlp', 'rnet_c1'])
def test_fp64_replays_the_oracle(name, swap_every):
    (layers, P), in_dim = NETS[name]
    G, nsteps = 2, 12
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 3, in_dim)
    assert prob.plan_info(8, True)['tensor_core'] == 0
    th0 = 0.5 * rs.randn(G, P)
    for method, mname in ((0, 'hmc'), (1, 'mala')):
        st, ps, recs = _pt(prob, th0, BETAS4, 0.02, nsteps, 17, G, method=mname, swap_every=swap_every)
        dev = _snapshot(st, ps, recs)
        eps = 0.02 / np.sqrt(BETAS4)
        ost, orec = _oracle(layers, x, y, 0.1, th0, nsteps, BETAS4, eps, method=method, swap_every=swap_every, seed=17)
        _compare(dev, ost, orec, G, nsteps, swap_every, 1e-9)
        assert ost['attempts'].sum() > 0


# ---------------------------------------------------------------------------------------------------------------- 3
@pytest.mark.parametrize('swap_every,split', [(1, 7), (3, 9)])
def test_runs_are_deterministic_split_and_resumable(swap_every, split):
    from quinn_b200 import ops
    layers, P = qo.mlp_layers(1, 1, (5, 4), True, 'tanh')
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 4, 1)
    G = 3
    th0 = 0.5 * rs.randn(G, P)
    kw = dict(betas=BETAS4, eps=0.03, nsteps=30, seed=9, G=G, swap_every=swap_every)
    a = _snapshot(*_pt(prob, th0, **kw))
    b = _snapshot(*_pt(prob, th0, **kw))
    c = _snapshot(*_pt(prob, th0, splits=(split,), **kw))
    assert a['swap_accepts'].sum() > 0
    for key in a:
        assert a[key].tobytes() == b[key].tobytes(), key
        assert a[key].tobytes() == c[key].tobytes(), key
    # resume from state_dicts into fresh objects
    st, ps, recs = _pt(prob, th0, BETAS4, 0.03, split, 9, G, swap_every=swap_every)
    sd, psd = st.state_dict(), ps.state_dict()
    st2 = ops.ChainState(prob, np.zeros((4 * G, P)))
    ps2 = ops.PtState(st2, G, BETAS4, 0.03, 3, 'hmc', swap_every)
    st2.load_state_dict(sd)
    ps2.load_state_dict(psd)
    rec = ops.Recorder(st2, 30 - split, store_every=1, sample_rows=G)
    ops.pt_run(st2, ps2, 30 - split, rec, seed=9)
    d = _snapshot(st2, ps2, [rec])
    for key in ('theta', 'lp', 'map_theta', 'map_lp', 'naccept', 'grad_cur', 'replica', 'last_end', 'round_trips',
                'swap_attempts', 'swap_accepts'):
        assert a[key].tobytes() == d[key].tobytes(), key
    assert a['logpost'][:, split:].tobytes() == d['logpost'].tobytes()


def test_thinned_records_match_one_call():
    """store_every a multiple of swap_every and the reverse: the cold draws land where qb_hmc_run would put them"""
    layers, P = qo.mlp_layers(1, 1, (5, 4), True, 'tanh')
    prob, x, y, rs = _problem(layers, P, 40, torch.float64, 4, 1)
    G = 2
    th0 = 0.5 * rs.randn(G, P)
    for swap_every, store_every in ((2, 6), (6, 2), (3, 3)):
        kw = dict(seed=5, G=G, swap_every=swap_every, store_every=store_every)
        got = _snapshot(*_pt(prob, th0, BETAS4, 0.03, 24, **kw))
        one = _snapshot(*_pt(prob, th0, BETAS4, 0.03, 24, seed=5, G=G, swap_every=swap_every))
        np.testing.assert_array_equal(got['samples'], one['samples'][:, store_every - 1::store_every])
        np.testing.assert_array_equal(got['logpost'], one['logpost'])
        assert got['samples'].shape == (G, 24 // store_every, P)


# ---------------------------------------------------------------------------------------------------------------- 4
def _group_close_step(orec, g, G, nsteps, tol):
    """the first step at which a chain of group g made an MH decision, or the group a swap decision, with margin <= tol"""
    K = orec['mh_margin'].shape[0]
    rows = list(range(g, K, G))
    for s in range(nsteps):
        if orec['mh_margin'][rows, s].min() <= tol:
            return s
        if min([m for gg, _, _, m in orec['swaps'][s] if gg == g] or [np.inf]) <= tol:
            return s
    return nsteps


@pytest.mark.parametrize('name', ['stream_f64', 'tcg_h32', 'tg8_h64', 'tg8_h128', 'cuda_f32'])
def test_every_path_agrees_with_the_oracle(name):
    """each group (its T chains are coupled by the swaps) is compared up to its first decision closer than a tenth of the
    path's tolerance"""
    _, (layers, P), in_dim, dtype, code, tol, eps = _path(name)
    G, nsteps = 8, 3
    T = len(BETAS4)
    prob, x, y, rs = _problem(layers, P, 64, dtype, 5, in_dim)
    assert prob.plan_info(T * G, True)['tensor_core'] == code
    th0 = _start(prob, rs, G, P, dtype)
    st, ps, recs = _pt(prob, th0, BETAS4, eps, nsteps, 31, G)
    dev = _snapshot(st, ps, recs)
    ost, orec = _oracle(layers, x, y, 0.1, th0, nsteps, BETAS4, eps / np.sqrt(BETAS4), seed=31)
    compared = 0
    for g in range(G):
        s_ok = _group_close_step(orec, g, G, nsteps, tol / 10)
        if s_ok == 0:
            continue
        compared += 1
        rows = list(range(g, T * G, G))
        lp = orec['lp'][rows, :s_ok]
        np.testing.assert_allclose(dev['logpost'][rows, :s_ok], lp, rtol=tol, atol=tol)
        np.testing.assert_array_equal(dev['accepted'][rows, :s_ok].astype(bool), orec['acc'][rows, :s_ok])
        cz = orec['cold_z'][:s_ok, g]
        assert np.abs(dev['samples'][g, :s_ok] - cz).max() <= tol * np.abs(cz).max(), g
    assert compared >= G // 2, compared


# ---------------------------------------------------------------------------------------------------------------- 5
def test_every_slot_samples_its_tempered_gaussian():
    """Linear(d, 1), flat prior: slot i targets N(theta_hat, sigma^2 (X~^T X~)^-1 / beta_i)"""
    from quinn_b200 import ops, post
    from quinn_b200.netdesc import netdesc_from_module
    d, N, sigma, G = 2, 200, 0.3, 512
    rs = np.random.RandomState(8)
    x = rs.randn(N, d)
    y = x @ rs.randn(d, 1) + 0.5 + sigma * rs.randn(N, 1)
    Xt = np.hstack([x, np.ones((N, 1))])
    cov = sigma ** 2 * np.linalg.inv(Xt.T @ Xt)
    mean = np.linalg.solve(Xt.T @ Xt, Xt.T @ y[:, 0])
    prob = ops.Problem(netdesc_from_module(torch.nn.Linear(d, 1)), x, y, sigma, dtype=torch.float64, device='cuda')
    betas = [1.0, 0.5, 0.25, 0.125]
    T = len(betas)
    eps = 0.5 * np.sqrt(np.linalg.eigvalsh(cov).min())
    st = ops.ChainState(prob, np.tile(mean + 0.05 * rs.randn(G, d + 1), (T, 1)))
    ps = ops.PtState(st, G, betas, eps, 3, 'hmc', 1)
    ops.pt_run(st, ps, 300, None, seed=4)
    n_keep = 400
    draws = torch.empty((n_keep, T * G, d + 1), dtype=torch.float64, device='cuda')
    for j in range(n_keep):
        ops.pt_run(st, ps, 2, None, seed=4)
        draws[j] = st.theta
    assert (ps.swap_accepts.sum() > 0.3 * ps.swap_attempts.sum()).item()
    for i, b in enumerate(betas):
        dr = draws[:, i * G:(i + 1) * G].transpose(0, 1)                    # [G, n_keep, P]
        for p in range(d + 1):
            for f, ref in ((dr[:, :, p], mean[p]), ((dr[:, :, p] - mean[p]) ** 2, cov[p, p] / b)):
                ess = post.ess(f.contiguous()).sum().item()
                se = f.std().item() / np.sqrt(ess)
                assert abs(f.mean().item() - ref) <= 5 * se, (i, p, f.mean().item(), ref, se, ess)


# ---------------------------------------------------------------------------------------------------------------- 6
def _two_mode_problem():
    """MLP(1, 1, (1,)) tanh with the prior sigma_p = 1, anchor 0: lp(w1, b1, w2, b2) = lp(-w1, -b1, -w2, b2) exactly"""
    from quinn_b200 import ops
    from quinn_b200.netdesc import netdesc_from_module
    from quinn_b200.nns import MLP
    rs = np.random.RandomState(1)
    N = 20
    x = np.linspace(-1, 1, N)[:, None]
    y = np.tanh(2 * x) + 0.3 * rs.randn(N, 1)
    net = MLP(1, 1, (1,), activ='tanh').double()
    desc = netdesc_from_module(net)
    prob = ops.Problem(desc, x, y, 0.5, dtype=torch.float64, device='cuda', prior_sigma=1.0,
                       prior_anchor=np.zeros(desc.n_params), fulldatasize=N)
    return prob, desc


def _w2_index(desc):
    return desc.layers[-1].w_off


def test_tempering_switches_between_the_two_modes():
    """Every group starts in the w2 > 0 mode (w1 = 2, w2 = 1).  The ladder (8 geometric temperatures down to 0.02),
    seeds and lengths are fixed.  On a B200 the pooled cold fraction with w2 < 0 after burn-in was 0.515 (bounds 0.35 and
    0.65), the 64 groups made 5324 round trips, and plain HMC at the same step size had a fraction of 0.0000 (bound
    0.01): it never left the start mode."""
    from quinn_b200 import ops
    prob, desc = _two_mode_problem()
    P, iw = desc.n_params, _w2_index(desc)
    G, burn, keep = 64, 1000, 3000
    th0 = np.zeros((G, P))
    th0[:, desc.layers[0].w_off] = 2.0
    th0[:, iw] = 1.0
    betas = ops.pt_ladder(8, 0.02)
    st = ops.ChainState(prob, np.tile(th0, (len(betas), 1)))
    ps = ops.PtState(st, G, betas, 0.05, 3, 'hmc', 1)
    ops.pt_run(st, ps, burn, None, seed=12)
    rec = ops.Recorder(st, keep, store_every=1, sample_rows=G)
    ops.pt_run(st, ps, keep, rec, seed=12)
    frac = (rec.samples[:, :, iw] < 0).double().mean().item()
    trips = ps.round_trips.sum().item()
    assert 0.35 <= frac <= 0.65, frac
    assert trips > 0
    st_h = ops.ChainState(prob, th0)
    hm = ops.HmcState(st_h, epsilon=0.05, L=3, method='hmc')
    rec_h = ops.Recorder(st_h, burn + keep, store_every=1)
    ops.hmc_run(st_h, hm, burn + keep, rec_h, seed=12)
    frac_h = (rec_h.samples[:, burn:, iw] < 0).double().mean().item()
    assert frac_h < 0.01, frac_h
    print(f'two modes: PT cold fraction w2 < 0 {frac:.3f}, round trips {trips}, HMC fraction {frac_h:.4f}')


# ---------------------------------------------------------------------------------------------------------------- 7
def _solver():
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_MCMC
    torch.manual_seed(3)
    rs = np.random.RandomState(3)
    x = rs.rand(50, 1) * 2 - 1
    return NN_MCMC(MLP(1, 1, (6,), activ='tanh').double(), verbose=False), x, np.sin(3 * x) + 0.1 * rs.randn(50, 1)


def test_solver_single_group_and_many_groups():
    from quinn_b200 import ops
    uq, x, y = _solver()
    P = uq.pdim
    sp = dict(epsilon=0.01, L=3, n_temps=4, beta_min=0.1)
    res = uq.fit(x, y, datanoise=0.1, nmcmc=20, sampler='pt', sampler_params=sp, seed=5)
    assert res['chain'].shape == (21, P) and res['logpost'].shape == (21,) and res['alphas'].shape == (21,)
    assert isinstance(res['maxpost'], float) and isinstance(res['accrate'], float)
    assert res['betas'].shape == (4,) and res['step_sizes'].shape == (4,) and res['swap_rate'].shape == (3,)
    assert isinstance(res['round_trips'], int)
    assert res['accrate'] == pytest.approx(res['accepted'].mean())
    assert uq.sampler_obj.last_state.K == 4
    res = uq.fit(x, y, datanoise=0.1, nmcmc=20, sampler='pt', sampler_params=dict(sp, base='mala', swap_every=2), seed=5,
                 nchains=3, zflag=False, store_every=2)
    assert res['chain'].shape == (3, 11, P) and res['logpost'].shape == (3, 21)
    assert res['swap_rate'].shape == (3, 3) and res['round_trips'].shape == (3,)
    assert uq.sampler_obj.last_state.K == 12
    # the cold log-posterior is the untempered one of the cold draws
    prob = uq.device_logpost(uq.lpinfo).problem
    lp = ops.logpost(prob, res['chain'][:, 1:].reshape(-1, P)).cpu().numpy().reshape(3, 10)
    np.testing.assert_allclose(res['logpost'][:, 2::2], lp, rtol=1e-12)
    d = uq.diagnose()
    assert d['ess_logpost'].shape == (3,)
    res = uq.fit(x, y, datanoise=0.1, nmcmc=10, sampler='pt', sampler_params=sp, seed=5, nchains=2, zflag=False,
                 keep_on_device=True)
    assert torch.is_tensor(res['chain']) and res['chain'].is_cuda and res['chain'].shape == (2, 11, P)
    assert torch.is_tensor(res['betas'])
    assert uq.predict_ens(x[:5], nens=2, nburn=2).shape == (4, 5, 1)


def test_solver_refusals():
    from quinn_b200.mcmc import PT
    uq, x, y = _solver()
    with pytest.raises(ValueError, match="'pt'"):
        uq.fit(x, y, nmcmc=3, sampler='pt', replay=dict(incr=np.zeros((3, uq.pdim)), unif=np.zeros(3)), zflag=False)
    for flag in ('distributed', 'data_sharded'):
        with pytest.raises(ValueError, match="'pt'"):
            uq.fit(x, y, nmcmc=3, sampler='pt', **{flag: True})
    m = PT()
    m.setLogPost(lambda th: -0.5 * float(np.sum(th ** 2)), None)
    with pytest.raises(ValueError, match='device log-posterior'):
        m.run(3, np.zeros(2), verbose=False)
