"""Layer-streamed kernels (quinn_b200/csrc/qb_stream.cuh): networks whose weights do not fit in shared memory next to one
tile of activations, through every entry point, against the oracle.  fp64: log-posterior 1e-10 relative, gradient 1e-9
of its largest entry; fp32: log-posterior 1e-4 relative, gradient 2e-3 of its largest entry."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_util import netdesc_from_layers
from oracle import quinn_oracle as qo

pytestmark = pytest.mark.gpu

F64, F32 = torch.float64, torch.float32


def _mlp(indim, outdim, hls, activ='tanh'):
    return qo.mlp_layers(indim, outdim, hls, True, activ)


# name -> (oracle layers, P, final transform, dtypes whose plan is streamed, theta scale)
NETS = {
    'mlp_160x2': (_mlp(10, 1, (160, 160)), None, (F64,), 0.08),
    'mlp_100x4': (_mlp(10, 1, (100, 100, 100, 100)), None, (F64,), 0.1),
    'mlp_128x3': (_mlp(10, 1, (128, 128, 128)), None, (F64,), 0.09),
    'rnet_128_poly1': (qo.rnet_layers(128, 3, 10, 1, poly_order=1), None, (F64, F32), 0.06),
    'mlp_256x2': (_mlp(10, 1, (256, 256)), None, (F64, F32), 0.06),
    'mlp_512x2': (_mlp(10, 1, (512, 512)), None, (F64, F32), 0.04),
    'mlp_256x3_relu_o2': (_mlp(5, 2, (256, 256, 256), 'relu'), None, (F64, F32), 0.06),
    'mlp_512x2_exp': (_mlp(3, 1, (512, 512)), 'exp', (F64, F32), 0.03),
    'rnet_256_poly0': (qo.rnet_layers(256, 2, 10, 1, shared=True), None, (F64, F32), 0.05),
}
CASES = [(n, dt) for n, v in NETS.items() for dt in v[2]]
IDS = [f'{n}-{"f64" if dt == F64 else "f32"}' for n, dt in CASES]


def _ops():
    from quinn_b200 import ops
    return ops


def _desc(name):
    (layers, P), final, _, _ = NETS[name]
    return layers, P, netdesc_from_layers(layers, P, final_exp=final == 'exp'), final


def _data(desc, N, seed):
    rs = np.random.RandomState(seed)
    x = rs.rand(N, desc.in_dim) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True) * np.arange(1, desc.out_dim + 1)[None, :]) + 0.1 * rs.randn(N, desc.out_dim)
    return x, y + (1.5 if desc.final_exp else 0.0)


def _thetas(K, P, scale, seed, dtype):
    g = torch.Generator(device='cuda').manual_seed(seed)
    return (scale * torch.randn((K, P), generator=g, device='cuda', dtype=F64)).to(dtype)


def _tols(dtype):
    return (1e-10, 1e-9) if dtype == F64 else (1e-4, 2e-3)


def _check_rows(layers, final, th, x, y, sigma, lp, gr, rows, dtype, prior=None, nfull=None):
    tol_lp, tol_g = _tols(dtype)
    for k in rows:
        pk = None if prior is None else dict(sigma=prior['sigma'], anchor=prior['anchor'][k])
        rl, rg = qo.logpost_grad(layers, th[k].double().cpu().numpy(), x, y, sigma, fulldatasize=nfull, prior=pk, final=final)
        assert abs(lp[k] - rl) <= tol_lp * abs(rl), (k, lp[k], rl)
        if gr is not None:
            err = np.abs(gr[k] - rg).max() / np.abs(rg).max()
            assert err <= tol_g, (k, err)


@pytest.mark.parametrize('name,dtype', CASES, ids=IDS)
def test_kernels_1_2_single_split_many_chains(name, dtype):
    ops = _ops()
    layers, P, desc, final = _desc(name)
    x, y = _data(desc, 150, 1)
    K = 2048
    th = _thetas(K, P, NETS[name][3], 2, dtype)
    kw = {}
    prior = None
    if name == 'mlp_256x3_relu_o2':               # per-chain prior anchors
        anchor = _thetas(K, P, 0.02, 3, dtype)
        kw = dict(prior_sigma=0.7, prior_anchor=anchor, fulldatasize=1000)
        prior = dict(sigma=0.7, anchor=anchor.double().cpu().numpy())
    prob = ops.Problem(desc, x, y, 0.2, dtype=dtype, **kw)
    for grad in (False, True):
        info = prob.plan_info(K, grad)
        assert info['tensor_core'] == 5 and info['splits'] == 1, info
    lp = ops.logpost(prob, th).cpu().numpy()
    lp2, gr = ops.logpost_grad(prob, th)
    rows = [0, 1, 777, K - 1]                      # a fixed subset of the chains
    grn = {k: gr[k].double().cpu().numpy() for k in rows}
    _check_rows(layers, final, th, x, y, 0.2, lp, None, rows, dtype, prior, 1000)
    _check_rows(layers, final, th, x, y, 0.2, lp2.cpu().numpy(), grn, rows, dtype, prior, 1000)


@pytest.mark.parametrize('name,dtype', CASES, ids=IDS)
def test_kernels_1_2_split_data_axis(name, dtype):
    ops = _ops()
    layers, P, desc, final = _desc(name)
    x, y = _data(desc, 3001, 4)
    K = 2
    th = _thetas(K, P, NETS[name][3], 5, dtype)
    prob = ops.Problem(desc, x, y, 0.3, dtype=dtype)
    for grad in (False, True):
        info = prob.plan_info(K, grad)
        assert info['tensor_core'] == 5 and info['splits'] > 1, info
    lp = ops.logpost(prob, th).cpu().numpy()
    lp2, gr = ops.logpost_grad(prob, th)
    lp2, gr = lp2.cpu().numpy(), gr.double().cpu().numpy()
    _check_rows(layers, final, th, x, y, 0.3, lp, None, range(K), dtype)
    _check_rows(layers, final, th, x, y, 0.3, lp2, gr, range(K), dtype)


@pytest.mark.parametrize('name', ['mlp_128x3', 'rnet_128_poly1', 'mlp_512x2_exp'])
def test_fp64_results_are_bit_identical_run_to_run(name):
    ops = _ops()
    layers, P, desc, final = _desc(name)
    x, y = _data(desc, 2000, 6)
    for K in (2, 300):
        th = _thetas(K, P, NETS[name][3], 7, F64)
        prob = ops.Problem(desc, x, y, 0.3, dtype=F64)
        a = [ops.logpost_grad(prob, th) for _ in range(2)]
        assert torch.equal(a[0][0], a[1][0]) and torch.equal(a[0][1], a[1][1])
        assert torch.equal(ops.logpost(prob, th), ops.logpost(prob, th))


@pytest.mark.parametrize('name,dtype', [('mlp_128x3', F64), ('mlp_256x3_relu_o2', F32), ('rnet_128_poly1', F64)])
def test_per_member_data(name, dtype):
    """qb_logpost_members: member k sees its own rows x[k], y[k] (strides n*d, n*o)."""
    from quinn_b200 import _lib
    from quinn_b200.ops import _ptr, _stream
    ops = _ops()
    layers, P, desc, final = _desc(name)
    K, n = 5, 300
    xs, ys = zip(*[_data(desc, n, 10 + k) for k in range(K)])
    x, y = np.concatenate(xs), np.concatenate(ys)
    th = _thetas(K, P, NETS[name][3], 8, dtype)
    prob = ops.Problem(desc, x, y, 0.25, dtype=dtype)
    lib = _lib.load()
    need = lib.qb_eval_workspace_bytes(C.byref(prob.cnet), prob.qdt, K, n, 1)
    assert need > 0
    ws = torch.empty(int(need), dtype=torch.uint8, device='cuda')
    data = _lib.qb_data_t(prob.x.data_ptr(), prob.y.data_ptr(), n)
    lp = torch.empty(K, dtype=F64, device='cuda')
    g = torch.empty((K, P), dtype=dtype, device='cuda')
    _lib.check(lib.qb_logpost_members(C.byref(prob.cnet), prob.qdt, _ptr(th), K, C.byref(data), n * desc.in_dim,
                                      n * desc.out_dim, C.byref(prob.clik), _ptr(lp), _ptr(g), _ptr(ws), ws.numel(),
                                      _stream()), 'qb_logpost_members')
    tol_lp, tol_g = _tols(dtype)
    lp, g = lp.cpu().numpy(), g.double().cpu().numpy()
    for k in range(K):
        rl, rg = qo.logpost_grad(layers, th[k].double().cpu().numpy(), xs[k], ys[k], 0.25, final=final)
        assert abs(lp[k] - rl) <= tol_lp * abs(rl)
        assert np.abs(g[k] - rg).max() <= tol_g * np.abs(rg).max()


def test_diagonal_fisher():
    from quinn_b200.nns import MLP, NNWrap, NegLogPost
    from quinn_b200.nns.tchutils import tch
    from quinn_b200.netdesc import netdesc_from_module, flatten_module
    torch.manual_seed(3)
    net = MLP(10, 1, (128, 128, 128), activ='tanh')
    desc = netdesc_from_module(net)
    layers = desc.as_oracle_layers()
    x, y = _data(desc, 24, 12)
    theta = flatten_module(net)
    anchor = 0.01 * np.random.RandomState(13).randn(theta.size)
    wrap = NNWrap(net)
    for prior in (None, {'sigma': 0.8, 'anchor': anchor}):
        loss = NegLogPost(wrap.nnmodel, 500, 0.1, None if prior is None else {'sigma': 0.8, 'anchor': tch(anchor)})
        f = wrap.calc_fisher_diag(theta, loss, x, y)
        ref = qo.diag_fisher(layers, theta, x, y, 0.1, fulldatasize=500, prior=prior)
        np.testing.assert_allclose(f, ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())


def _replay_setup(name, nsteps, seed):
    ops = _ops()
    layers, P, desc, final = _desc(name)
    x, y = _data(desc, 200, seed)
    rs = np.random.RandomState(seed)
    th0 = NETS[name][3] * rs.randn(1, P)
    prob = ops.Problem(desc, x, y, 0.2, dtype=F64)
    st = ops.ChainState(prob, th0)
    rec = ops.Recorder(st, nsteps, store_every=1)
    u = rs.rand(nsteps)
    unif = torch.as_tensor(u, dtype=F64, device='cuda').reshape(nsteps, 1).contiguous()
    return ops, layers, P, final, x, y, th0, prob, st, rec, rs, u, unif


def _check_chain(st, rec, ref):
    acc = rec.accepted[0].cpu().numpy().astype(bool)
    assert np.array_equal(acc, ref['accepted']), np.nonzero(acc != ref['accepted'])[0][:5]
    assert acc.sum() > 0
    np.testing.assert_allclose(rec.samples[0].cpu().numpy(), ref['chain'][1:], rtol=1e-10, atol=1e-13)
    np.testing.assert_allclose(rec.logpost[0].cpu().numpy(), ref['logpost'][1:], rtol=1e-10)
    np.testing.assert_allclose(st.theta[0].cpu().numpy(), ref['chain'][-1], rtol=1e-10, atol=1e-13)


@pytest.mark.parametrize('method', ['hmc', 'mala'])
def test_hmc_and_mala_replay(method):
    nsteps = 30
    ops, layers, P, final, x, y, th0, prob, st, rec, rs, u, unif = _replay_setup('mlp_128x3', nsteps, 21)
    assert prob.plan_info(1, True)['tensor_core'] == 5
    p = rs.randn(nsteps, P)
    eps = 4e-4 if method == 'hmc' else 3e-4
    hm = ops.HmcState(st, method=method, epsilon=eps, L=3)
    ops.hmc_run(st, hm, nsteps, rec, incr=torch.as_tensor(p, device='cuda').reshape(nsteps, 1, P).contiguous(), unif=unif)
    torch.cuda.synchronize()
    lpf = lambda th: qo.logpost(layers, th, x, y, 0.2, final=final)            # noqa: E731
    gf = lambda th: qo.logpost_grad(layers, th, x, y, 0.2, final=final)[1]     # noqa: E731
    ref = qo.run_chain(lpf, th0[0], nsteps, method, dict(p=p, u=u), grad_fn=gf, epsilon=eps, L=3)
    _check_chain(st, rec, ref)


def test_amcmc_replay():
    nsteps = 30
    ops, layers, P, final, x, y, th0, prob, st, rec, rs, u, unif = _replay_setup('mlp_128x3', nsteps, 22)
    assert prob.plan_info(1, False)['tensor_core'] == 5
    xi = 2e-3 * rs.randn(nsteps, P)
    am = ops.AmcmcState(st, adapt='none', t0=10 * nsteps)
    ops.amcmc_run(st, am, nsteps, rec, incr=torch.as_tensor(xi, device='cuda').reshape(nsteps, 1, P).contiguous(), unif=unif)
    torch.cuda.synchronize()
    # the accept loop of MCMCBase.run (mcmc.py:69-85) with the increments supplied
    cur = th0[0].copy()
    lp_cur = qo.logpost(layers, cur, x, y, 0.2, final=final)
    chain, lps, accs = [cur.copy()], [lp_cur], []
    for t in range(nsteps):
        prop = cur + xi[t]
        lp_prop = qo.logpost(layers, prop, x, y, 0.2, final=final)
        with np.errstate(over='ignore'):
            acc = bool(u[t] < np.exp(lp_prop - lp_cur))
        if acc:
            cur, lp_cur = prop, lp_prop
        chain.append(cur.copy()); lps.append(lp_cur); accs.append(acc)
    _check_chain(st, rec, dict(accepted=np.array(accs), chain=np.array(chain), logpost=np.array(lps)))


@pytest.mark.parametrize('name,dtype', [('mlp_512x2_exp', F64), ('mlp_256x3_relu_o2', F32), ('rnet_128_poly1', F64),
                                        ('mlp_128x3', F64)])
def test_predictive(name, dtype):
    ops = _ops()
    layers, P, desc, final = _desc(name)
    x, _ = _data(desc, 1000, 30)
    M = 6
    th = _thetas(M, P, NETS[name][3], 31, dtype)
    ref = qo.predict_ens(layers, th.double().cpu().numpy(), x, final=final)
    out, mean, var = ops.predict(desc, th, x, dtype=dtype, want_out=True, want_moments=True)
    tol = 1e-11 if dtype == F64 else 2e-5
    scale = np.abs(ref).max()
    np.testing.assert_allclose(out.double().cpu().numpy(), ref, rtol=tol, atol=tol * scale)
    np.testing.assert_allclose(mean.double().cpu().numpy(), ref.mean(0), rtol=tol, atol=tol * scale)
    np.testing.assert_allclose(var.double().cpu().numpy(), ref.var(0, ddof=1), rtol=1e3 * tol, atol=tol * scale ** 2)
    # moments only (no `out` buffer from the caller)
    o2, mean2, var2 = ops.predict(desc, th, x, dtype=dtype, want_out=False, want_moments=True)
    assert o2 is None
    assert torch.equal(mean2, mean) and torch.equal(var2, var)


def _solver_data():
    rs = np.random.RandomState(40)
    x = rs.rand(128, 10) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(128, 1)
    return x, y


@pytest.mark.parametrize('sampler,params', [('amcmc', {}), ('hmc', {'epsilon': 1e-4, 'L': 3})])
def test_nn_mcmc_many_chains(sampler, params):
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_MCMC
    np.random.seed(41)
    torch.manual_seed(41)
    net = MLP(10, 1, (128, 128, 128), activ='tanh')
    x, y = _solver_data()
    uq = NN_MCMC(net, verbose=False)
    res = uq.fit(x, y, zflag=False, datanoise=0.1, nmcmc=1010, sampler=sampler, sampler_params=params, nchains=8,
                 seed=5, keep_on_device=True)
    lp = torch.as_tensor(res['logpost']).cpu().numpy()
    assert lp.shape == (8, 1011) and np.all(np.isfinite(lp)) and torch.as_tensor(res['accrate']).shape == (8,)
    xt = np.random.rand(9, 10) * 2 - 1
    m, v, _ = uq.predict_mom_sample(xt, msc=1, nsam=5)
    assert m.shape == (9, 1) and v.shape == (9, 1) and np.all(np.isfinite(m)) and np.all(np.isfinite(v))


def test_nn_ens_batched():
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_Ens
    from quinn_b200.netdesc import flatten_module, netdesc_from_module
    np.random.seed(42)
    torch.manual_seed(42)
    net = MLP(10, 1, (128, 128, 128), activ='tanh')
    x, y = _solver_data()
    ens = NN_Ens(net, nens=3, dfrac=0.8)
    layers = netdesc_from_module(net).as_oracle_layers()
    before = [np.mean((qo.forward(layers, flatten_module(l.nnmodel), x) - y) ** 2) for l in ens.learners]
    ens.fit(x, y, nepochs=8, lrate=0.002, freq_out=1000)
    assert ens.batched_fit and np.all(np.isfinite(ens.fit_info['best_loss']))
    after = [np.mean((qo.forward(layers, flatten_module(l.best_model), x) - y) ** 2) for l in ens.learners]
    assert all(a < b for a, b in zip(after, before)), (before, after)
    assert np.all(np.isfinite(ens.predict_ens(x[:7])))


def test_nn_vi():
    from quinn_b200.nns import MLP
    from quinn_b200.solvers import NN_VI
    np.random.seed(43)
    torch.manual_seed(43)
    net = MLP(10, 1, (128, 128, 128), activ='tanh')
    x, y = _solver_data()
    vi = NN_VI(net, verbose=False, seed=4)
    vi.fit(x, y, nepochs=12, lrate=0.01, nsam=4, datanoise=0.1, freq_out=1000)
    hist = np.array(vi.fit_info['history'])
    assert np.all(np.isfinite(hist[:, 3]))
    assert hist[-3:, 3].mean() < hist[:3, 3].mean()
    assert np.all(np.isfinite(vi.predict_ens(x[:5], nens=3)))
