"""The adapted-proposal branches of the fused AMCMC kernels (admcmc.py:52-70), driven PAST adaptation points.

* Philox mode, fp64, CUDA-core kernel: the device chain is replayed step by step on the CPU with oracle/philox.py (the
  counter-based streams restated in numpy, pinned to the Random123 known-answer vectors) and the oracle's run_chain, both
  for the diagonal adaptation (the repo's scalable deviation, DESIGN.md section 5) and for the initial rank-1 + diagonal
  proposal; chain, decisions, running mean / covariance and proposal scales must agree.
* fp32 tensor-core kernels k_amcmc_tc3 (config-5 shape) and k_amcmc<float,2> (other eligible shapes): replay mode
  across adaptation points against the oracle recursion, and Philox mode against the CUDA-core kernel run from the same
  seed (identical proposals => identical chains up to fp32-noise ties), which exercises the kind == 1 proposal branch.
* the in-kernel Cholesky survives a rank-deficient covariance (first adaptation with fewer samples than parameters).
"""
import numpy as np
import pytest
import torch

from golden_util import netdesc_from_layers
from oracle import philox
from oracle import quinn_oracle as qo
from test_gpu_tensorcore import make_net, no_tc

pytestmark = pytest.mark.gpu


def _problem(widths, N, seed, dtype, sigma=0.3):
    from quinn_b200 import ops
    rs = np.random.RandomState(seed)
    layers, P = make_net(widths, ['tanh', 'tanh', 'identity'])
    x = rs.rand(N, widths[0]) * 2 - 1
    y = np.sin(x.sum(1, keepdims=True)) + 0.05 * rs.randn(N, 1)
    prob = ops.Problem(netdesc_from_layers(layers, P), x, y, sigma, dtype=dtype)
    return rs, layers, P, x, y, prob


def test_philox_numpy_restatement_known_answers():
    """oracle/philox.py against the published Philox4x32-10 known-answer vectors; the device generator is then pinned to
    the numpy restatement by the chain replays below (any difference in a single word changes a proposal)."""
    # known answers of Philox4x32-10 (Random123 kat_vectors): the numpy restatement is pinned here, the device to it below
    assert [int(v) for v in philox.philox4x32_10((0, 0, 0, 0), (0, 0))] == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert [int(v) for v in philox.philox4x32_10((0xffffffff,) * 4, (0xffffffff,) * 2)] == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]


@pytest.mark.parametrize('seed,chain_offset', [(11, 0), (2 ** 40 + 5, 123456789012)])
def test_amcmc_diag_adaptation_fp64_replayed_with_numpy_philox(seed, chain_offset):
    from quinn_b200 import ops
    rs, layers, P, x, y, prob = _problem([2, 8, 8, 1], 60, 5, torch.float64)
    K, steps, gamma, t0, tadapt = 3, 75, 0.3, 10, 20
    th0 = 0.4 * rs.randn(K, P)
    st = ops.ChainState(prob, th0)
    am = ops.AmcmcState(st, gamma=gamma, t0=t0, tadapt=tadapt, adapt='diag')
    rec = ops.Recorder(st, steps, store_every=1)
    ops.amcmc_run(st, am, steps, rec, seed=seed, chain_offset=chain_offset)
    torch.cuda.synchronize()
    lpf = lambda th: qo.logpost(layers, th, x, y, 0.3)                 # noqa: E731
    for k in range(K):
        draws = philox.amcmc_draws(seed, chain_offset + k, steps, P)
        ref = qo.run_chain(lpf, th0[k], steps, 'amcmc', draws, gamma=gamma, t0=t0, tadapt=tadapt)
        assert ref['_kind'] == 1                                     # the run went through adaptations
        assert np.array_equal(rec.accepted[k].cpu().numpy().astype(bool), ref['accepted'])
        assert 0.05 < ref['accepted'].mean() < 0.99
        np.testing.assert_allclose(rec.samples[k].cpu().numpy(), ref['chain'][1:], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(rec.logpost[k].cpu().numpy(), ref['logpost'][1:], rtol=1e-10)
        np.testing.assert_allclose(am.xm[k].cpu().numpy(), ref['_Xm'], rtol=1e-10, atol=1e-13)
        np.testing.assert_allclose(am.cov[k].cpu().numpy(), np.diag(ref['_cov']), rtol=1e-8, atol=1e-14)
        np.testing.assert_allclose(am.pscale[k].cpu().numpy(), ref['_pscale'], rtol=1e-8)
        assert int(am.prop_kind[k].item()) == 1


@pytest.mark.parametrize('widths,tc_kind', [([3, 64, 64, 1], 'hot'), ([2, 32, 32, 1], 'general')])
def test_tc_amcmc_replay_across_adaptation_points(widths, tc_kind):
    """k_amcmc_tc3 / k_amcmc<float,2> with adapt='diag' in replay mode, 70 steps with t0=10, tadapt=20: decisions, chain and
    the adapted proposal scales against the oracle recursion."""
    from quinn_b200 import ops
    rs, layers, P, x, y, prob = _problem(widths, 300, 7, torch.float32)
    assert prob.plan_info(4)['tensor_core'] == 2
    K, steps, gamma, t0, tadapt = 3, 70, 0.2, 10, 20
    th0 = (0.3 * rs.randn(K, P)).astype(np.float32).astype(np.float64)
    incr = (0.004 * rs.randn(steps, K, P)).astype(np.float32).astype(np.float64)
    u = rs.rand(steps, K)
    st = ops.ChainState(prob, th0)
    am = ops.AmcmcState(st, gamma=gamma, t0=t0, tadapt=tadapt, adapt='diag')
    rec = ops.Recorder(st, steps, store_every=1)
    ops.amcmc_run(st, am, steps, rec, incr=torch.as_tensor(incr, dtype=torch.float32, device='cuda'), unif=torch.as_tensor(u, device='cuda'))
    torch.cuda.synchronize()
    lpf = lambda th: qo.logpost(layers, th, x, y, 0.3)                 # noqa: E731
    fac = gamma * 2.4 ** 2 / P
    for k in range(K):
        ref = qo.run_chain(lpf, th0[k], steps, 'amcmc', dict(xi=incr[:, k], u=u[:, k]), gamma=gamma, t0=t0, tadapt=tadapt)
        acc = rec.accepted[k].cpu().numpy().astype(bool)
        same = acc == ref['accepted']
        if not same.all():                                           # only a tie at fp32 noise may differ
            first = int(np.where(~same)[0][0])
            assert abs(u[first, k] - ref['alphas'][1 + first]) <= 1e-3
            continue
        assert 0.1 < acc.mean() < 1.0
        np.testing.assert_allclose(rec.samples[k].double().cpu().numpy(), ref['chain'][1:], rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(rec.logpost[k].cpu().numpy(), ref['logpost'][1:], rtol=2e-5)
        np.testing.assert_allclose(am.xm[k].double().cpu().numpy(), ref['_Xm'], rtol=1e-4, atol=1e-6)
        np.testing.assert_allclose(am.cov[k].double().cpu().numpy(), np.diag(ref['_cov']), rtol=2e-3, atol=1e-10)
        # the scales in force at the end were computed at the last adaptation (step 60) from the covariance of that step;
        # replay the recursion up to there
        Xm = cov = None
        for t in range(61):
            Xm, cov = qo.amcmc_moments_update(Xm, cov, ref['chain'][t], t)
        np.testing.assert_allclose(am.pscale[k].double().cpu().numpy(), np.sqrt(fac * (np.diag(cov) + 1e-8)), rtol=2e-3)
        assert int(am.prop_kind[k].item()) == 1


@pytest.mark.parametrize('widths', [[3, 64, 64, 1], [2, 32, 32, 1]])
def test_tc_amcmc_philox_adapted_proposals_equal_the_cuda_core_kernel(widths):
    """Philox mode across adaptation points: the tensor-core kernels (kind == 1 branch of the proposal in k_amcmc_tc3
    and of qb_amcmc_pre in k_amcmc<float,2>) and the CUDA-core kernel draw the same proposals, so states agree wherever decisions agree."""
    from quinn_b200 import ops
    rs, layers, P, x, y, prob = _problem(widths, 400, 9, torch.float32, sigma=0.5)
    K, steps = 48, 70
    th0 = rs.rand(K, P)

    def run():
        st = ops.ChainState(prob, th0)
        am = ops.AmcmcState(st, gamma=0.05, t0=10, tadapt=20, adapt='diag')
        rec = ops.Recorder(st, steps, store_every=1)
        ops.amcmc_run(st, am, steps, rec, seed=31)
        torch.cuda.synchronize()
        return st, am, rec

    st, am, rec = run()
    assert prob.plan_info(K)['tensor_core'] == 2
    with no_tc():
        assert prob.plan_info(K)['tensor_core'] == 0
        st2, am2, rec2 = run()
    a1, a2 = rec.accepted.cpu().numpy().astype(bool), rec2.accepted.cpu().numpy().astype(bool)
    assert (a1 != a2).mean() < 0.01
    assert 0.02 < a1[:, 21:].mean() < 0.98                  # adapted proposals get accepted and rejected
    same = (a1 == a2).all(axis=1)
    assert same.sum() >= K // 2
    s1, s2 = rec.samples.cpu().numpy(), rec2.samples.cpu().numpy()
    np.testing.assert_allclose(s1[same], s2[same], rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(am.pscale.cpu().numpy()[same], am2.pscale.cpu().numpy()[same], rtol=1e-5)
    assert (am.prop_kind.cpu().numpy() == 1).all()
    # after the last adaptation the accepted moves are pscale * z: finite, non-zero, of the adapted size
    moved = np.abs(s1[:, 65] - s1[:, 60]).max(axis=1)
    assert np.isfinite(s1).all() and (moved[a1[:, 61:66].any(axis=1)] > 0).all()
    # the recorded log-posteriors are the oracle's at the stored states
    for k in (0, K - 1):
        ref = qo.logpost(layers, s1[k, steps - 1].astype(np.float64), x, y, 0.5)
        assert abs(rec.logpost[k, steps - 1].item() - ref) <= 1e-5 * abs(ref)


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_full_adaptation_survives_a_rank_deficient_covariance(dtype):
    """adapt='full' with the first adaptation after 12 steps of a P = 105 chain: the covariance has rank <= 12; the
    in-kernel Cholesky must not produce NaN proposals (the reference draws through an SVD and tolerates PSD matrices,
    admcmc.py:70)."""
    from quinn_b200 import ops
    rs, layers, P, x, y, prob = _problem([2, 8, 8, 1], 50, 13, dtype)
    K, steps = 4, 60
    th0 = 0.3 * rs.randn(K, P)
    with no_tc():
        st = ops.ChainState(prob, th0)
        am = ops.AmcmcState(st, gamma=0.5, t0=5, tadapt=12, adapt='full')
        rec = ops.Recorder(st, steps, store_every=1)
        ops.amcmc_run(st, am, steps, rec, seed=3)
        torch.cuda.synchronize()
    assert torch.isfinite(am.chol).all()
    assert torch.isfinite(rec.samples).all() and torch.isfinite(rec.logpost).all()
    acc = rec.accepted.cpu().numpy().astype(bool)
    assert acc[:, 13:].any()                               # proposals from the adapted factor are accepted at times
    Lf = am.chol[0].double().cpu().numpy()
    cov = am.cov[0].double().cpu().numpy()
    assert (np.diag(Lf) > 0).all()
    # the factor in force was computed at step 48 (the covariance kept moving afterwards): check it is a valid factor of a
    # PSD matrix of the right scale rather than an exact identity
    fac = 0.5 * 2.4 ** 2 / P
    assert np.abs(Lf @ Lf.T).max() <= 50 * fac * (np.abs(cov).max() + 1e-8)
