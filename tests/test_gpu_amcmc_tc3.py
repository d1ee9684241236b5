"""k_amcmc_tc3, the hot-shape fp32 AMCMC chain kernel (quinn_b200/csrc/qb_value_tc3.cu), replayed step by step against
the numpy restatement of tests/chain_replay.py, and the edges of the warp-specialised value kernels (qb_tc3.cuh).

A  flat posterior: every proposal is accepted, so the recorded chain IS the proposal sequence; on k_amcmc_tc3,
   k_amcmc<float, 2> and the CUDA-core fp32 kernel, across t0 and three adaptation points, with a chain offset >= 2^32,
   and at the two chains of seed 2026 whose draws hit the extreme 24-bit uniforms (u1 = 1 - 2^-23 and u1 = 1).
B  a real posterior, every step of every chain checked given the device's own previous state: N from 1 to 10^4
   (1 to 79 tiles), both x-staging variants, input widths 1 to 7, missing biases, a tanh output layer, priors with
   shared and per-chain anchors, thinned records.
C  bit identity across launch splits and between a chain run alone and inside a 200-chain launch.
D  the value kernels at width 128, near chunk boundaries, with degenerate and badly scaled W1 and with saturating
   proposals inside the chain kernel; tolerances from the error model of qb_tc3.cuh.
"""
import math
import os

import numpy as np
import pytest
import torch

import chain_replay as cr
from golden_util import netdesc_from_layers
from oracle import philox
from oracle import quinn_oracle as qo

pytestmark = pytest.mark.gpu

HOT_THREADS = 288                      # 8 compute warps + the issue warp: the plan of k_logpost_tc3 / k_amcmc_tc3


class env:
    """Set library switches (read at every launch) for the enclosed calls."""
    def __init__(self, **kw):
        self.kw = kw

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kw}
        os.environ.update({k: str(v) for k, v in self.kw.items()})

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                del os.environ[k]
            else:
                os.environ[k] = v


def net(in_dim=3, width=64, bias=(True, True, True), out_act='identity'):
    widths, acts = [in_dim, width, width, 1], ['tanh', 'tanh', out_act]
    layers, off = [], 0
    for l in range(3):
        w = off
        off += widths[l] * widths[l + 1]
        b = -1
        if bias[l]:
            b = off
            off += widths[l + 1]
        layers.append(dict(n_in=widths[l], n_out=widths[l + 1], w_off=w, b_off=b, act=acts[l], res_step=0.0))
    return layers, off


def staging(K, P, N):
    """Which x staging k_amcmc_tc3 uses (qb_tc3_launch_amcmc): bulk tiles in the proposal scratch when K P floats hold
    the ceil(N / 128) split tiles of 8 KiB, else the compute threads stage each tile."""
    return 'bulk' if K * P * 4 >= ((N + 127) // 128) * 8192 else 'compute'


class Case:
    def __init__(self, layers, P, N, sigma, seed, prior=None, fulldatasize=None, anchor_per_chain=None, K=1):
        from quinn_b200 import ops
        rs = np.random.RandomState(seed)
        self.layers, self.P, self.N, self.sigma = layers, P, N, sigma
        d = layers[0]['n_in']
        self.x = rs.rand(N, d) * 2 - 1
        self.y = np.sin(self.x.sum(1, keepdims=True)) + 0.05 * rs.randn(N, 1)
        self.rs = rs
        self.prior_sigma, self.full = prior, fulldatasize
        self.anchor = None
        kw = {}
        if prior is not None:
            self.anchor = (0.1 * rs.randn(K, P) if anchor_per_chain else 0.1 * rs.randn(P)).astype(np.float32)
            kw = dict(prior_sigma=prior, prior_anchor=self.anchor, fulldatasize=fulldatasize)
        self.prob = ops.Problem(netdesc_from_layers(layers, P), self.x, self.y, sigma, dtype=torch.float32, **kw)

    def lpg(self, k):
        prior = None
        if self.prior_sigma is not None:
            prior = dict(sigma=self.prior_sigma, anchor=(self.anchor[k] if self.anchor.ndim == 2 else self.anchor).astype(np.float64))
        return lambda th: qo.logpost_grad(self.layers, th, self.x, self.y, self.sigma, self.full, prior)


def run(prob, th0, steps, adapt='diag', seed=1, chain_offset=0, gamma=0.2, t0=5, tadapt=10, store_every=1, splits=None):
    from quinn_b200 import ops
    st = ops.ChainState(prob, th0)
    am = ops.AmcmcState(st, gamma=gamma, t0=t0, tadapt=tadapt, adapt=adapt)
    recs = []
    for n in (splits or [steps]):
        rec = ops.Recorder(st, n, store_every=store_every)
        ops.amcmc_run(st, am, n, rec, seed=seed, chain_offset=chain_offset)
        recs.append(rec)
    torch.cuda.synchronize()
    return st, am, recs


def chain_rec(st, am, recs, k):
    g = lambda t: t[k].cpu().numpy()                     # noqa: E731
    cat = lambda name: np.concatenate([getattr(r, name)[k].cpu().numpy() for r in recs])     # noqa: E731
    return dict(samples=cat('samples'), logpost=cat('logpost'), alpha=cat('alpha'), accepted=cat('accepted'),
                logpost0=float(recs[0].logpost0[k]), lp=float(st.lp[k]), theta=g(st.theta), map_lp=float(st.map_lp[k]),
                map_theta=g(st.map_theta), naccept=int(st.naccept[k]), xm=None if am.xm is None else g(am.xm),
                cov=None if am.cov is None else g(am.cov), pscale=g(am.pscale), prop_kind=int(am.prop_kind[k]))


def check_chains(case, st, am, recs, th0, steps, ks, seed, chain_offset=0, gamma=0.2, t0=5, tadapt=10, adapt='diag',
                 **kw):
    """check_amcmc_steps on chains ks; a recorded log-posterior may deviate by 1e-5 relative or, where cancellation
    makes |lp| small (N = 1), by the error model's bound (lp_bound below)."""
    lp_tol = lambda th: max(1e-5 * abs(qo.logpost(case.layers, th, case.x, case.y, case.sigma)),       # noqa: E731
                            lp_bound(case.layers, th, case.x, case.y, case.sigma))
    out = []
    for k in ks:
        draws = cr.amcmc_draws_f32(seed, chain_offset + k, steps, case.P)
        rec = chain_rec(st, am, recs, k)
        out.append((rec, cr.check_amcmc_steps(rec, th0[k], draws, case.lpg(k), gamma, t0, tadapt, adapt, lp_tol=lp_tol,
                                              **kw)))
    return out


def report(tag, results):
    """One line per case with the chain-steps checked and the largest deviation / tolerance of each check."""
    m = {key: max(r[1][key] for r in results) for key in ('lp', 'proposal', 'log_alpha')}
    n = sum(r[1]['steps'] for r in results)
    print(f'[amcmc_tc3 margins] {tag}: chain-steps {n}  lp {m["lp"]:.3g}  proposal {m["proposal"]:.3g}  '
          f'log_alpha {m["log_alpha"]:.3g}')


# ---- A: flat posterior ------------------------------------------------------------------------------------------------
A_KERNELS = {
    'tc3': ([3, 64, 64, 1], {}, lambda i: i['threads'] == HOT_THREADS),
    'tc2-hot-shape': ([3, 64, 64, 1], dict(QB_NO_V3=1), lambda i: i['tensor_core'] == 2 and i['threads'] != HOT_THREADS),
    'tc2-2-32-32-1': ([2, 32, 32, 1], {}, lambda i: i['tensor_core'] == 2 and i['threads'] != HOT_THREADS),
    'cuda-core': ([3, 64, 64, 1], dict(QB_NO_TC=1), lambda i: i['tensor_core'] == 0),
}


@pytest.mark.parametrize('kernel', list(A_KERNELS))
def test_flat_posterior_chain_is_the_restated_proposal_sequence(kernel):
    widths, sw, plan_ok = A_KERNELS[kernel]
    layers, P = net(widths[0], widths[1])
    case = Case(layers, P, 50, 1e9, 3)
    K, steps, seed, off, t0, tadapt = 3, 70, 99, 2 ** 32 + 5, 10, 20
    th0 = (0.3 * case.rs.randn(K, P)).astype(np.float32)
    with env(**sw):
        assert plan_ok(case.prob.plan_info(K)), case.prob.plan_info(K)
        st, am, recs = run(case.prob, th0, steps, seed=seed, chain_offset=off, t0=t0, tadapt=tadapt)
    res = check_chains(case, st, am, recs, th0, steps, range(K), seed, off, t0=t0, tadapt=tadapt)
    for rec, _ in res:
        assert rec['accepted'].all() and rec['prop_kind'] == 1
    report(f'A {kernel}', res)


@pytest.mark.parametrize('chain,step,block,m', [(1459, 3, 410, 2 ** 24 - 2), (2654, 1, 247, 2 ** 24 - 1)])
def test_draws_at_the_extreme_uniforms_are_finite(chain, step, block, m):
    """The bench seed's chains whose radius word z gives u1 = 1 - 2^-23 (ln u1 = -1.19e-7, below __logf's absolute
    error) and u1 = 1 (ln u1 = 0): the two normals of that word must be finite (a NaN would reject the step silently)."""
    layers, P = net(3)
    case = Case(layers, P, 1, 1e9, 4)
    seed = 2026
    w = philox.rand4(seed, chain, step, philox.STREAM_INCR, np.array([block]))
    assert int(w[2][0] >> 8) == m                                 # the word is the one the restatement says
    th0 = (0.3 * case.rs.randn(1, P)).astype(np.float32)
    assert case.prob.plan_info(1)['threads'] == HOT_THREADS
    st, am, recs = run(case.prob, th0, 5, seed=seed, chain_offset=chain)
    res = check_chains(case, st, am, recs, th0, 5, [0], seed, chain)
    rec = res[0][0]
    assert rec['accepted'].all() and np.isfinite(rec['samples']).all()
    i = 4 * block + 2
    prev = rec['samples'][step - 1] if step else th0[0]
    kind_draws = cr.amcmc_draws_f32(seed, chain, 5, P)
    ps = np.sqrt(0.09 * np.abs(th0[0].astype(np.float64))).astype(np.float32)
    z_dev = (rec['samples'][step][i:i + 2].astype(np.float64) - prev[i:i + 2] - kind_draws['z0'][step]) / ps[i:i + 2]
    print(f'[amcmc_tc3 extreme uniform] chain {chain} step {step} params {i}-{i + 1}: device z ~ {z_dev}, '
          f'restated {kind_draws["z"][step][i:i + 2]} +- {kind_draws["z_err"][step][i:i + 2]}')
    report(f'A extreme chain {chain}', res)


# ---- B: per-step replay with a real posterior ------------------------------------------------------------------------
B_CASES = {
    'N1': dict(N=1, K=1, adapt='diag', staging='bulk'),
    'N100': dict(N=100, K=2, adapt='none', staging='bulk'),
    'N128': dict(N=128, K=1, adapt='diag', staging='bulk'),
    'N129': dict(N=129, K=2, adapt='none', staging='bulk'),
    'N256': dict(N=256, K=1, adapt='diag', staging='bulk'),
    'N257-compute': dict(N=257, K=1, adapt='diag', staging='compute'),
    'N385-compute': dict(N=385, K=1, adapt='none', staging='compute'),
    'N385-bulk': dict(N=385, K=3, adapt='diag', staging='bulk'),
    'N10000-compute': dict(N=10000, K=2, adapt='diag', staging='compute'),
    'N10000-bulk': dict(N=10000, K=40, adapt='diag', staging='bulk', ks=(0, 39)),
    'in1': dict(in_dim=1, N=300, K=2),
    'in4': dict(in_dim=4, N=300, K=2),
    'in7': dict(in_dim=7, N=300, K=2),
    'in7-compute': dict(in_dim=7, N=700, K=1, staging='compute'),
    'no-bias0': dict(bias=(False, True, True), N=300, K=2),
    'no-bias1': dict(bias=(True, False, True), N=300, K=2),
    'no-bias2': dict(bias=(True, True, False), N=300, K=2),
    'tanh-output': dict(out_act='tanh', N=300, K=2),
    'prior-shared': dict(N=300, K=2, prior=0.7, full=1500),
    'prior-per-chain': dict(N=300, K=3, prior=1.3, full=150, per_chain=True),
}
B_STEPS = 30


def _b_case(name):
    c = dict(in_dim=3, bias=(True, True, True), out_act='identity', adapt='diag', prior=None, full=None, per_chain=None)
    c.update(B_CASES[name])
    layers, P = net(c['in_dim'], bias=c['bias'], out_act=c['out_act'])
    sigma = 0.3 * math.sqrt(c['N'])              # keeps the log-ratios of the first proposals finite and non-zero
    case = Case(layers, P, c['N'], sigma, 17, c['prior'], c['full'], c['per_chain'], c['K'])
    th0 = (0.05 * case.rs.randn(c['K'], P)).astype(np.float32)
    return c, case, th0


@pytest.mark.parametrize('name', list(B_CASES))
def test_replay_every_step_against_the_restatement(name):
    c, case, th0 = _b_case(name)
    K, P, N = c['K'], case.P, case.N
    assert case.prob.plan_info(K)['threads'] == HOT_THREADS
    if 'staging' in c:
        assert staging(K, P, N) == c['staging']
    st, am, recs = run(case.prob, th0, B_STEPS, adapt=c['adapt'], seed=5)
    res = check_chains(case, st, am, recs, th0, B_STEPS, c.get('ks', range(K)), 5, adapt=c['adapt'])
    acc = np.concatenate([r[0]['accepted'] for r in res]).astype(bool)
    assert acc.any() and not acc.all()
    report(f'B {name} ({staging(K, P, N)} staging, T = {(N + 127) // 128})', res)


def test_thinned_records_hold_every_third_state():
    c, case, th0 = _b_case('N385-bulk')
    _, _, r1 = run(case.prob, th0, B_STEPS, seed=5)
    _, _, r3 = run(case.prob, th0, B_STEPS, seed=5, store_every=3)
    s1, s3 = r1[0].samples.cpu().numpy(), r3[0].samples.cpu().numpy()
    assert s3.shape[1] == B_STEPS // 3
    assert np.array_equal(s3.view(np.uint32), s1[:, 2::3].view(np.uint32))
    for name in ('logpost', 'alpha', 'accepted'):
        assert torch.equal(getattr(r1[0], name), getattr(r3[0], name))


# ---- C: bit identity ------------------------------------------------------------------------------------------------
def _state_arrays(st, am):
    return dict(theta=st.theta, lp=st.lp, naccept=st.naccept, map_theta=st.map_theta, map_lp=st.map_lp, xm=am.xm,
                cov=am.cov, pscale=am.pscale, prop_kind=am.prop_kind)


@pytest.mark.parametrize('N', [100, 200, 10000])
def test_launch_splits_are_bit_identical(N):
    layers, P = net(3)
    case = Case(layers, P, N, 0.3 * math.sqrt(N), 23)
    K = 3
    th0 = (0.05 * case.rs.randn(K, P)).astype(np.float32)
    st1, am1, r1 = run(case.prob, th0, B_STEPS, seed=8)
    st2, am2, r2 = run(case.prob, th0, B_STEPS, seed=8, splits=[1, 1, 7, B_STEPS - 9])     # crosses t0 = 5 and t = 10
    for name, a in _state_arrays(st1, am1).items():
        assert torch.equal(a, _state_arrays(st2, am2)[name]), name
    for name in ('logpost', 'alpha', 'accepted', 'samples'):
        whole = getattr(r1[0], name)
        assert torch.equal(whole, torch.cat([getattr(r, name) for r in r2], dim=1)), name
    assert torch.equal(r1[0].logpost0, r2[0].logpost0)


@pytest.mark.parametrize('N', [100, 200, 10000])
def test_chain_alone_equals_the_chain_among_200(N):
    layers, P = net(3)
    case = Case(layers, P, N, 0.3 * math.sqrt(N), 29)
    K, j = 200, 137
    th0 = (0.05 * case.rs.randn(K, P)).astype(np.float32)
    st1, am1, r1 = run(case.prob, th0, B_STEPS, seed=8)
    st2, am2, r2 = run(case.prob, th0[j:j + 1], B_STEPS, seed=8, chain_offset=j)
    if N == 10000:
        assert staging(K, P, N) == 'bulk' and staging(1, P, N) == 'compute'
    for name, a in _state_arrays(st1, am1).items():
        assert torch.equal(a[j:j + 1], _state_arrays(st2, am2)[name]), name
    for name in ('logpost', 'alpha', 'accepted', 'samples', 'logpost0'):
        assert torch.equal(getattr(r1[0], name)[j:j + 1], getattr(r2[0], name)), name


# ---- D: value-kernel edges ----------------------------------------------------------------------------------------------
# Error model (qb_tc3.cuh): layer 0 in 3xTF32 and the hidden GEMM in 3xFP16 carry ~22 significant bits per product;
# W1's fp16 lo parts below 2^-16 of the largest entry carry an absolute error of 2^-25 of the scaled maximum (taken
# here as 2^-24 max|W1| per entry); activations come from ex2 / rcp approximations and fp16 hi/lo pairs (~2^-22).
E_PROD, E_ACT, E_W1 = 2.0 ** -21, 2.0 ** -21, 2.0 ** -24


def out_bound(layers, th, x):
    """Per-point bound on |out_device - out_exact| for an in -> H -> H -> 1 tanh net under the error model."""
    (W0, b0), (W1, b1), (W2, b2) = [qo._layer_wb(L, np.asarray(th, np.float64)) for L in layers]
    b0 = np.zeros(W0.shape[0]) if b0 is None else b0
    b1 = np.zeros(W1.shape[0]) if b1 is None else b1
    b2 = np.zeros(1) if b2 is None else b2
    z0 = x @ W0.T + b0
    a0 = np.tanh(z0)
    e0 = E_PROD * (np.abs(x) @ np.abs(W0).T + np.abs(b0)) + E_ACT
    z1 = a0 @ W1.T + b1
    a1 = np.tanh(z1)
    e1 = e0 @ np.abs(W1).T + E_PROD * (np.abs(a0) @ np.abs(W1).T + np.abs(b1)) + W1.shape[1] * E_W1 * np.abs(W1).max() + E_ACT
    e2 = e1 @ np.abs(W2).T + E_PROD * (np.abs(a1) @ np.abs(W2).T + np.abs(b2))
    if layers[2]['act'] == 'tanh':
        e2 = e2 + E_ACT
    return e2[:, 0]


def lp_bound(layers, th, x, y, sigma):
    """|lp_device - lp_exact| <= sum |r| e / s^2 + sum e^2 / (2 s^2) + 2^-20 ssq / (2 s^2) (fp32 residuals and sums)."""
    r = y[:, 0] - qo.forward(layers, th, x)[:, 0]
    e = out_bound(layers, th, x)
    return (np.sum(np.abs(r) * e) + 0.5 * np.sum(e * e) + 2.0 ** -20 * 0.5 * np.sum(r * r)) / sigma ** 2


def _value_check(layers, P, th, x, y, sigma, threads):
    from quinn_b200 import ops
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, sigma, dtype=torch.float32)
    assert prob.plan_info(th.shape[0])['threads'] == threads
    lp = ops.logpost(prob, th).cpu().numpy()
    out, _, _ = ops.predict(prob.desc, th, x, dtype=torch.float32)
    worst = 0.0
    for k in range(th.shape[0]):
        ref = qo.logpost(layers, th[k].astype(np.float64), x, y, sigma)
        b = lp_bound(layers, th[k], x, y, sigma)
        assert abs(lp[k] - ref) <= b, (k, lp[k], ref, b)
        eo = out_bound(layers, th[k], x)
        d = np.abs(out[k, :, 0].double().cpu().numpy() - qo.forward(layers, th[k].astype(np.float64), x)[:, 0])
        assert np.all(d <= eo), (k, d.max(), eo[np.argmax(d - eo)])
        worst = max(worst, abs(lp[k] - ref) / b, float(np.max(d / eo)))
    return worst


@pytest.mark.parametrize('variant', ['plain', 'zero-W1', 'one-W1-entry-1e3'])
@pytest.mark.parametrize('width,in_dim', [(64, 7), (128, 15)])
def test_value_kernels_within_the_error_model(width, in_dim, variant):
    rs = np.random.RandomState(41)
    layers, P = net(in_dim, width)
    N, M = 1000, 3
    x = rs.rand(N, in_dim) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(N, 1)
    th = (rs.randn(M, P) / np.sqrt(width)).astype(np.float32)
    w1 = slice(layers[1]['w_off'], layers[1]['w_off'] + width * width)
    if variant == 'zero-W1':
        th[:, w1] = 0.0
    elif variant == 'one-W1-entry-1e3':
        th[:, layers[1]['w_off'] + 5 * width + 9] *= 1e3
    worst = _value_check(layers, P, th, x, y, 0.2, 128 * (width // 32) + 32)
    print(f'[amcmc_tc3 margins] D value width {width} in {in_dim} {variant}: worst deviation / bound {worst:.3g}')


def test_predict_near_chunk_boundaries():
    """Few members: blocks hold one or two tiles, N one point either side of a chunk boundary (qb_tile_chunks)."""
    from quinn_b200 import ops
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    layers, P = net(3)
    desc = netdesc_from_layers(layers, P)
    rs = np.random.RandomState(43)
    for M in (1, 2):
        chunks = -(-sms * 16 // M)                     # blocks wanted per member
        for N in (chunks * 128 - 1, chunks * 128 + 1):           # one tile per block / two
            x = rs.rand(N, 3) * 2 - 1
            th = (rs.randn(M, P) / 8).astype(np.float32)
            out, _, _ = ops.predict(desc, th, x, dtype=torch.float32)
            o = out.double().cpu().numpy()[:, :, 0]
            for m in range(M):
                ref = qo.forward(layers, th[m].astype(np.float64), x)[:, 0]
                assert np.all(np.abs(o[m] - ref) <= out_bound(layers, th[m], x)), (M, N, m)


def test_chain_kernel_with_saturating_proposals():
    """Proposals whose layer 0 saturates (|W0| ~ 10^3) and whose W1 has one entry 10^3 times the rest: the chain
    kernel's per-proposal W1 scaling (wmax) and the saturated epilogue, every step against the restatement with the
    log-posterior tolerance of the error model."""
    layers, P = net(3)
    case = Case(layers, P, 300, 30.0, 47)
    K = 2
    th0 = (0.05 * case.rs.randn(K, P)).astype(np.float32)
    th0[:, :3 * 64] *= 2e4
    th0[:, layers[1]['w_off'] + 64 * 7 + 3] = 50.0
    assert case.prob.plan_info(K)['threads'] == HOT_THREADS
    st, am, recs = run(case.prob, th0, B_STEPS, seed=6)
    res = []
    for k in range(K):
        draws = cr.amcmc_draws_f32(6, k, B_STEPS, P)
        rec = chain_rec(st, am, recs, k)
        tol = lambda th: lp_bound(layers, th, case.x, case.y, case.sigma)          # noqa: E731
        res.append((rec, cr.check_amcmc_steps(rec, th0[k], draws, case.lpg(k), 0.2, 5, 10, 'diag', lp_tol=tol)))
    acc = np.concatenate([r[0]['accepted'] for r in res]).astype(bool)
    assert acc.any()
    report('D saturating chain', res)
