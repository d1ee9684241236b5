"""Torch-tensor front end of the C ABI (include/quinn_b200.h).

PyTorch is used here only for device memory and streams; every computation is a call into
libquinn_b200.so through ctypes.  All functions require CUDA tensors and raise otherwise.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from .netdesc import NetDesc


def qb_dtype(dtype):
    if dtype == torch.float32:
        return _lib.QB_F32
    if dtype == torch.float64:
        return _lib.QB_F64
    raise TypeError(f'quinn_b200 computes in float32 or float64, not {dtype}')


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError('quinn_b200 kernels need CUDA tensors (there is no CPU fallback)')


def as_device(a, dtype, device):
    """numpy / tensor -> contiguous tensor of `dtype` on `device`."""
    if isinstance(a, list):
        a = np.array(a)
    t = torch.as_tensor(a)
    return t.to(device=device, dtype=dtype, non_blocking=True).contiguous()     # async from pinned host memory


class Problem:
    """Network + data + likelihood resident on one GPU: everything kernels 1-3 need besides theta.

    Mirrors what the reference re-creates on every evaluation (nn_mcmc.py:55-66: a fresh NNWrap, NegLogPost
    and torch.tensor copies of x and y); here it is built once.
    """

    def __init__(self, desc: NetDesc, x, y, sigma, dtype=torch.float32, device='cuda', prior_sigma=None,
                 prior_anchor=None, fulldatasize=None):
        self.desc = desc
        self.dtype = dtype
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('quinn_b200 needs a CUDA device (there is no CPU fallback)')
        self.qdt = qb_dtype(dtype)
        self.x = as_device(x, dtype, self.device)
        self.y = as_device(y, dtype, self.device)
        if self.x.dim() != 2 or self.y.dim() != 2 or self.x.shape[0] != self.y.shape[0]:
            raise ValueError('x must be (N,d) and y (N,o) with the same N')
        if self.x.shape[1] != desc.in_dim or self.y.shape[1] != desc.out_dim:
            raise ValueError(f'data dims {self.x.shape[1]}->{self.y.shape[1]} do not match the network '
                             f'{desc.in_dim}->{desc.out_dim}')
        self.n = int(self.x.shape[0])
        self.sigma = float(sigma)
        self.cnet = desc.to_c()
        self.cdata = _lib.qb_data_t(self.x.data_ptr(), self.y.data_ptr(), self.n)
        self.anchor = None
        self.clik = _lib.qb_lik_t()
        self.clik.sigma = self.sigma
        self.clik.prior_sigma = -1.0
        self.clik.prior_scale = 0.0
        if prior_sigma is not None:
            self.clik.prior_sigma = float(prior_sigma)
            full = self.n if fulldatasize is None else fulldatasize
            self.clik.prior_scale = float(self.n) / float(full)           # losses.py:204
            if prior_anchor is not None:
                self.anchor = as_device(prior_anchor, dtype, self.device)
                self.clik.prior_anchor = self.anchor.data_ptr()
                self.clik.anchor_per_chain = 1 if self.anchor.dim() == 2 else 0
        self._ws = {}

    def workspace(self, K, want_grad):
        key = (K, bool(want_grad))
        ws = self._ws.get(key)
        if ws is None:
            lib = _lib.load()
            nbytes = lib.qb_eval_workspace_bytes(C.byref(self.cnet), self.qdt, K, self.n, 1 if want_grad else 0)
            if nbytes == 0:
                _lib.check(-1, 'qb_eval_workspace_bytes')
            ws = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
            self._ws = {key: ws}          # keep only the latest shape
        return ws

    def plan_info(self, K, want_grad=False):
        out = (C.c_int64 * 8)()
        _lib.check(_lib.load().qb_plan_info(C.byref(self.cnet), self.qdt, K, self.n, 1 if want_grad else 0, out),
                   'qb_plan_info')
        return dict(TM=out[0], threads=out[1], smem_bytes=out[2], splits=out[3], blocks=out[4], inplace=out[5],
                    tensor_core=int(out[6]), tmem_cols=int(out[7]))

    def theta(self, theta):
        t = as_device(theta, self.dtype, self.device)
        if t.dim() == 1:
            t = t[None, :]
        if t.shape[1] != self.desc.n_params:
            raise ValueError(f'theta has {t.shape[1]} parameters, the network has {self.desc.n_params}')
        return t.contiguous()


def logpost(prob: Problem, theta, out=None):
    """Kernel 1: lp[K] (float64, CUDA) for theta[K,P]."""
    theta = prob.theta(theta)
    _need_cuda(theta)
    K = theta.shape[0]
    lp = out if out is not None else torch.empty(K, dtype=torch.float64, device=prob.device)
    ws = prob.workspace(K, False)
    with torch.cuda.device(prob.device):
        rc = _lib.load().qb_logpost(C.byref(prob.cnet), prob.qdt, _ptr(theta), K, C.byref(prob.cdata), C.byref(prob.clik),
                                    _ptr(lp), _ptr(ws), ws.numel(), _stream())
    _lib.check(rc, 'qb_logpost')
    return lp


def logpost_grad(prob: Problem, theta, lp=None, grad=None):
    """Kernel 2: (lp[K] float64, grad[K,P] dtype)."""
    theta = prob.theta(theta)
    K = theta.shape[0]
    if lp is None:
        lp = torch.empty(K, dtype=torch.float64, device=prob.device)
    if grad is None:
        grad = torch.empty_like(theta)
    ws = prob.workspace(K, True)
    with torch.cuda.device(prob.device):
        rc = _lib.load().qb_logpost_grad(C.byref(prob.cnet), prob.qdt, _ptr(theta), K, C.byref(prob.cdata),
                                         C.byref(prob.clik), _ptr(lp), _ptr(grad), _ptr(ws), ws.numel(), _stream())
    _lib.check(rc, 'qb_logpost_grad')
    return lp, grad


def hvp_plan_info(prob: Problem, K):
    """Launch plan of kernel 5 for K directions; raises for a network the kernel refuses."""
    out = (C.c_int64 * 8)()
    _lib.check(_lib.load().qb_hvp_plan_info(C.byref(prob.cnet), prob.qdt, K, prob.n, out), 'qb_hvp_plan_info')
    return dict(TM=out[0], threads=out[1], smem_bytes=out[2], splits=out[3], blocks=out[4])


def _hvp(prob: Problem, theta, v, col0, K, out):
    if prob.clik.anchor_per_chain:
        raise ValueError('Hessian-vector products are taken at one theta: the prior anchor must be a single vector')
    lib = _lib.load()
    nbytes = lib.qb_hvp_workspace_bytes(C.byref(prob.cnet), prob.qdt, K, prob.n)
    if nbytes == 0 and K > 0:
        hvp_plan_info(prob, K)            # raises with the reason when the network is refused
    ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=prob.device)
    with torch.cuda.device(prob.device):
        rc = lib.qb_logpost_hvp(C.byref(prob.cnet), prob.qdt, _ptr(theta), _ptr(v), int(col0), int(K), C.byref(prob.cdata),
                                C.byref(prob.clik), _ptr(out), _ptr(ws), ws.numel(), _stream())
    _lib.check(rc, 'qb_logpost_hvp')
    return out


def logpost_hvp(prob: Problem, theta, v):
    """Kernel 5: hv[K,P] = (d^2 lp / d theta^2) v_k at one theta[P], for directions v[K,P] (or v[P])."""
    theta = prob.theta(theta)
    if theta.shape[0] != 1:
        raise ValueError('logpost_hvp takes a single theta')
    v = prob.theta(v)
    return _hvp(prob, theta, v, 0, v.shape[0], torch.empty_like(v))


def logpost_hessian(prob: Problem, theta, block=None):
    """Full Hessian d^2 lp / d theta^2 [P,P] on the device, filled by blocks of `block` unit directions (default: all P
    in one launch; kernel 5 caps its N-split workspace at 256 MB)."""
    theta = prob.theta(theta)
    if theta.shape[0] != 1:
        raise ValueError('logpost_hessian takes a single theta')
    P = prob.desc.n_params
    block = P if block is None else int(block)
    if block < 1:
        raise ValueError('block must be positive')
    H = torch.empty((P, P), dtype=prob.dtype, device=prob.device)
    for c0 in range(0, P, block):
        K = min(block, P - c0)
        _hvp(prob, theta, None, c0, K, H[c0:c0 + K])
    return H


def kfac_plan_info(prob: Problem):
    """Launch plan of kernel 6 over the problem's points; raises for a network the kernel refuses."""
    out = (C.c_int64 * 8)()
    _lib.check(_lib.load().qb_kfac_plan_info(C.byref(prob.cnet), prob.qdt, prob.n, out), 'qb_kfac_plan_info')
    return dict(TM=out[0], threads=out[1], smem_bytes=out[2], splits=out[3], factor_elems=out[4])


def kfac_layout(desc: NetDesc):
    """Per layer (n_in, n_out, has_bias, offset of A, offset of s or -1, offset of G) in kernel 6's factor row."""
    out, off = [], 0
    for L in desc.layers:
        a_off = off
        off += L.n_in * L.n_in
        s_off = off if L.b_off >= 0 else -1
        off += L.n_in if L.b_off >= 0 else 0
        out.append((L.n_in, L.n_out, L.b_off >= 0, a_off, s_off, off))
        off += L.n_out * L.n_out
    return out


def logpost_kfac(prob: Problem, theta):
    """Kernel 6: per layer dict(A, s, G) of float64 device tensors at one theta[P] -- the raw sums over the data points
    A = sum_i a_i a_i^T [n_in, n_in], s = sum_i a_i [n_in] (None without a bias), G = sum_i delta_i delta_i^T
    [n_out, n_out], with a_i the layer's input and delta_i = d log p_i / d z of point i's data term."""
    theta = prob.theta(theta)
    if theta.shape[0] != 1:
        raise ValueError('logpost_kfac takes a single theta')
    if prob.clik.anchor_per_chain:
        raise ValueError('Kronecker factors are taken at one theta: the prior anchor must be a single vector')
    F = kfac_plan_info(prob)['factor_elems']            # raises with the reason when the network is refused
    lib = _lib.load()
    fac = torch.empty(F, dtype=torch.float64, device=prob.device)
    nbytes = lib.qb_kfac_workspace_bytes(C.byref(prob.cnet), prob.qdt, prob.n)
    ws = torch.empty(max(int(nbytes), 1), dtype=torch.uint8, device=prob.device)
    with torch.cuda.device(prob.device):
        rc = lib.qb_logpost_kfac(C.byref(prob.cnet), prob.qdt, _ptr(theta), C.byref(prob.cdata), C.byref(prob.clik),
                                 _ptr(fac), _ptr(ws), ws.numel(), _stream())
    _lib.check(rc, 'qb_logpost_kfac')
    out = []
    for n_in, n_out, bias, a_off, s_off, g_off in kfac_layout(prob.desc):
        out.append(dict(A=fac[a_off:a_off + n_in * n_in].view(n_in, n_in),
                        s=fac[s_off:s_off + n_in] if bias else None,
                        G=fac[g_off:g_off + n_out * n_out].view(n_out, n_out)))
    return out


def jac_plan_info(desc: NetDesc, N, dtype=torch.float32):
    """Launch plan of kernel 7 over N points; raises for a network the kernel refuses.  rows = F, the factor rows of N
    elements each."""
    out = (C.c_int64 * 8)()
    cnet = desc.to_c()
    _lib.check(_lib.load().qb_jac_plan_info(C.byref(cnet), qb_dtype(dtype), int(N), out), 'qb_jac_plan_info')
    return dict(TM=out[0], threads=out[1], smem_bytes=out[2], blocks=out[3], rows=out[4])


def predict_jac(desc: NetDesc, theta, x, dtype=torch.float32, device='cuda'):
    """Kernel 7: f[N, o] at one theta[P] and, per layer, dict(a=[n_in, N], d=[o, n_out, N]) with a the layer's input and
    d[j] = d f_j / d z its pre-activation gradient (views into one buffer).  Layer l's part of d f_j(x_n) / d [W_l | b_l]
    is outer(d[j, :, n], [a[:, n]; 1])."""
    device = torch.device(device)
    theta = as_device(theta, dtype, device)
    if theta.dim() == 2 and theta.shape[0] == 1:
        theta = theta[0]
    x = as_device(x, dtype, device)
    _need_cuda(theta, x)
    if theta.dim() != 1 or theta.shape[0] != desc.n_params or x.dim() != 2 or x.shape[1] != desc.in_dim:
        raise ValueError('predict_jac takes a single theta[P] and x[N, in_dim] that match the network')
    N, o = x.shape[0], desc.out_dim
    F = jac_plan_info(desc, N, dtype)['rows']          # raises with the reason when the network is refused
    out = torch.empty((N, o), dtype=dtype, device=device)
    fac = torch.empty(N * F, dtype=dtype, device=device)
    cnet = desc.to_c()
    with torch.cuda.device(device):
        rc = _lib.load().qb_predict_jac(C.byref(cnet), qb_dtype(dtype), _ptr(theta), _ptr(x), N, _ptr(out), _ptr(fac),
                                        _stream())
    _lib.check(rc, 'qb_predict_jac')
    pairs, row = [], 0
    for L in desc.layers:
        a = fac[row * N:(row + L.n_in) * N].view(L.n_in, N)
        row += L.n_in
        d = fac[row * N:(row + o * L.n_out) * N].view(o, L.n_out, N)
        row += o * L.n_out
        pairs.append(dict(a=a, d=d))
    return out, pairs


def predict(desc: NetDesc, theta, x, dtype=torch.float32, device='cuda', want_out=True, want_moments=False,
            cnet=None):
    """Kernel 4: theta[M,P], x[N,d] -> out[M,N,o] and/or (mean[N,o], var[N,o], ddof=1)."""
    device = torch.device(device)
    theta = as_device(theta, dtype, device)
    if theta.dim() == 1:
        theta = theta[None, :]
    x = as_device(x, dtype, device)
    _need_cuda(theta, x)
    M, N, o = theta.shape[0], x.shape[0], desc.out_dim
    if theta.shape[1] != desc.n_params or x.shape[1] != desc.in_dim:
        raise ValueError('theta / x do not match the network')
    # moments of many members: run member-parallel (weights staged once per block) into a scratch array and reduce it
    # with k_moments, unless the scratch would be huge; then fall back to the fused per-tile member loop
    scratch = want_moments and not want_out and M > 1 and M * N * o * theta.element_size() <= 16 * 2 ** 30
    out = torch.empty((M, N, o), dtype=dtype, device=device) if (want_out or scratch) else None
    mean = torch.empty((N, o), dtype=dtype, device=device) if want_moments else None
    var = torch.empty((N, o), dtype=dtype, device=device) if want_moments else None
    cnet = cnet if cnet is not None else desc.to_c()
    lib = _lib.load()
    with torch.cuda.device(device):
        rc = lib.qb_predict(C.byref(cnet), qb_dtype(dtype), _ptr(theta), M, _ptr(x), N, _ptr(out), _ptr(mean), _ptr(var),
                            _stream())
        if rc != 0 and want_moments and not want_out:
            # moments of very wide outputs need the member-parallel path: give it an out buffer
            out = torch.empty((M, N, o), dtype=dtype, device=device)
            rc = lib.qb_predict(C.byref(cnet), qb_dtype(dtype), _ptr(theta), M, _ptr(x), N, _ptr(out), _ptr(mean),
                                _ptr(var), _stream())
            out = None
    _lib.check(rc, 'qb_predict')
    return (out if want_out else None), mean, var


class ChainState:
    """Device arrays of K chains (qb_chain_t) + per-sampler scratch."""

    def __init__(self, prob: Problem, theta0):
        self.prob = prob
        self.theta = prob.theta(theta0).clone()
        K, P = self.theta.shape
        dev = prob.device
        self.K, self.P = K, P
        self.lp = torch.zeros(K, dtype=torch.float64, device=dev)
        self.naccept = torch.zeros(K, dtype=torch.int64, device=dev)
        self.map_theta = torch.empty_like(self.theta)
        self.map_lp = torch.zeros(K, dtype=torch.float64, device=dev)
        self.t = 0                 # absolute step counter
        self.initialised = False

    def c(self):
        return _lib.qb_chain_t(self.K, self.theta.data_ptr(), self.lp.data_ptr(), self.naccept.data_ptr(),
                               self.map_theta.data_ptr(), self.map_lp.data_ptr())

    # checkpoint / resume (SURVEY.md section 5): Philox is counter based, so (state, seed, t) resumes exactly
    _FIELDS = ('theta', 'lp', 'naccept', 'map_theta', 'map_lp')

    def state_dict(self):
        d = {k: getattr(self, k).detach().cpu().clone() for k in self._FIELDS}
        d.update(t=self.t, initialised=self.initialised)
        return d

    def load_state_dict(self, d):
        for k in self._FIELDS:
            getattr(self, k).copy_(d[k])
        self.t, self.initialised = int(d['t']), bool(d['initialised'])


def _rng_struct(seed, chain_offset, incr, unif):
    r = _lib.qb_rng_t()
    if incr is not None:
        r.mode = _lib.QB_RNG_REPLAY
        r.incr = incr.data_ptr()
        r.unif = unif.data_ptr()
    else:
        r.mode = _lib.QB_RNG_PHILOX
    r.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    r.chain_offset = int(chain_offset)
    return r


class Recorder:
    """Per-step records of one run segment (qb_record_t)."""

    def __init__(self, state: ChainState, nsteps, store_every=1, record_scalars=True):
        dev, K, P = state.prob.device, state.K, state.P
        self.nsteps = nsteps
        self.store_every = int(store_every)
        self.n_slots = nsteps // self.store_every if self.store_every > 0 else 0
        self.logpost = torch.empty((K, nsteps), dtype=torch.float64, device=dev) if record_scalars else None
        self.alpha = torch.empty((K, nsteps), dtype=torch.float64, device=dev) if record_scalars else None
        self.accepted = torch.empty((K, nsteps), dtype=torch.uint8, device=dev) if record_scalars else None
        self.samples = (torch.empty((K, self.n_slots, P), dtype=state.prob.dtype, device=dev)
                        if self.n_slots > 0 else None)
        self.logpost0 = torch.empty(K, dtype=torch.float64, device=dev)     # filled by the first segment of a run

    def c(self):
        r = _lib.qb_record_t()
        if self.logpost is not None:
            r.logpost, r.alpha, r.accepted = self.logpost.data_ptr(), self.alpha.data_ptr(), self.accepted.data_ptr()
        r.ld = self.nsteps
        if self.samples is not None:
            r.samples = self.samples.data_ptr()
        r.store_every = self.store_every
        r.n_slots = self.n_slots
        r.logpost0 = self.logpost0.data_ptr()
        return r


class AmcmcState:
    """qb_amcmc_t: running mean / covariance / proposal factors of K chains (admcmc.py:34-36)."""

    def __init__(self, state: ChainState, gamma=0.1, t0=100, tadapt=1000, adapt='none', track=0, chol_ini=None):
        prob, K, P = state.prob, state.K, state.P
        dev, dt = prob.device, prob.dtype
        self.adapt = {'none': _lib.QB_ADAPT_NONE, 'diag': _lib.QB_ADAPT_DIAG, 'full': _lib.QB_ADAPT_FULL}[adapt]
        self.track = {'none': track, 'diag': 1, 'full': 2}[adapt]
        self.gamma, self.t0, self.tadapt = float(gamma), int(t0), int(tadapt)
        self.xm = torch.zeros((K, P), dtype=dt, device=dev) if self.track else None
        self.cov = None
        if self.track == 1:
            self.cov = torch.zeros((K, P), dtype=dt, device=dev)
        elif self.track == 2:
            if K * P * P * prob.x.element_size() > 8 * 2 ** 30:
                raise MemoryError(f"adapt='full' needs K*P*P = {K * P * P} covariance entries; use adapt='diag'")
            self.cov = torch.zeros((K, P, P), dtype=dt, device=dev)
        self.chol = torch.zeros((K, P, P), dtype=dt, device=dev) if self.adapt == _lib.QB_ADAPT_FULL else None
        self.pscale = torch.zeros((K, P), dtype=dt, device=dev)
        self.chol_ini = as_device(chol_ini, dt, dev) if chol_ini is not None else None
        self.prop_kind = torch.zeros(K, dtype=torch.int32, device=dev)
        self.scratch = torch.empty((K, P), dtype=dt, device=dev)

    _FIELDS = ('xm', 'cov', 'pscale', 'chol', 'prop_kind')

    def state_dict(self):
        return {k: getattr(self, k).detach().cpu().clone() for k in self._FIELDS if getattr(self, k) is not None}

    def load_state_dict(self, d):
        for k, v in d.items():
            getattr(self, k).copy_(v)

    def c(self):
        a = _lib.qb_amcmc_t()
        a.gamma, a.t0, a.tadapt, a.adapt, a.track_moments = self.gamma, self.t0, self.tadapt, self.adapt, self.track
        for name in ('xm', 'cov', 'pscale', 'chol', 'chol_ini', 'prop_kind'):
            t = getattr(self, name)
            if t is not None:
                setattr(a, name, t.data_ptr())
        return a


def amcmc_run(state: ChainState, am: AmcmcState, nsteps, rec: Recorder = None, seed=0, chain_offset=0, incr=None,
              unif=None):
    """Kernel 3 (AMCMC): advance all chains by nsteps; incr/unif given -> replay the reference's draws."""
    prob = state.prob
    rng = _rng_struct(seed, chain_offset, incr, unif)
    cch, cam = state.c(), am.c()
    crec = rec.c() if rec is not None else None
    with torch.cuda.device(prob.device):
        rc = _lib.load().qb_amcmc_run(C.byref(prob.cnet), prob.qdt, C.byref(prob.cdata), C.byref(prob.clik), C.byref(cch),
                                      C.byref(cam), C.byref(rng), C.byref(crec) if crec is not None else None,
                                      state.t, nsteps, 0 if state.initialised else 1, _ptr(am.scratch), _stream())
    _lib.check(rc, 'qb_amcmc_run')
    state.t += nsteps
    state.initialised = True


class HmcState:
    """qb_hmc_t: cached gradient + leapfrog scratch of K chains."""

    def __init__(self, state: ChainState, epsilon=0.05, L=3, method='hmc'):
        self.method = {'hmc': 0, 'mala': 1}[method]
        self.epsilon, self.L = float(epsilon), int(L)
        self.grad_cur = torch.zeros_like(state.theta)
        self.mom = torch.zeros_like(state.theta)
        self.prop = torch.zeros_like(state.theta)
        self.grad_prop = torch.zeros_like(state.theta)

    def state_dict(self):
        return dict(grad_cur=self.grad_cur.detach().cpu().clone())

    def load_state_dict(self, d):
        self.grad_cur.copy_(d['grad_cur'])

    def c(self):
        return _lib.qb_hmc_t(self.method, self.L, self.epsilon, self.grad_cur.data_ptr(), self.mom.data_ptr(),
                             self.prop.data_ptr(), self.grad_prop.data_ptr())


def hmc_run(state: ChainState, hm: HmcState, nsteps, rec: Recorder = None, seed=0, chain_offset=0, incr=None,
            unif=None):
    """Kernel 3 (HMC / MALA)."""
    prob = state.prob
    rng = _rng_struct(seed, chain_offset, incr, unif)
    cch, chm = state.c(), hm.c()
    crec = rec.c() if rec is not None else None
    with torch.cuda.device(prob.device):
        rc = _lib.load().qb_hmc_run(C.byref(prob.cnet), prob.qdt, C.byref(prob.cdata), C.byref(prob.clik), C.byref(cch),
                                    C.byref(chm), C.byref(rng), C.byref(crec) if crec is not None else None,
                                    state.t, nsteps, 0 if state.initialised else 1, _stream())
    _lib.check(rc, 'qb_hmc_run')
    state.t += nsteps
    state.initialised = True


def vi_sample(mu, rho, nsam, pi, sigma1, sigma2, eps=None, seed=0, step=0):
    """w[nsam,P] = mu + exp(rho)*eps, log q[nsam], log prior[nsam] (bnet.py:142-166)."""
    _need_cuda(mu, rho)
    P = mu.numel()
    dt, dev = mu.dtype, mu.device
    if eps is None:
        if not seed:
            raise ValueError('vi_sample needs eps or a non-zero seed')
        eps = torch.empty((nsam, P), dtype=dt, device=dev)
        use_seed = int(seed)
    else:
        eps = as_device(eps, dt, dev)
        use_seed = 0
    w = torch.empty((nsam, P), dtype=dt, device=dev)
    logq = torch.empty(nsam, dtype=torch.float64, device=dev)
    logp = torch.empty(nsam, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        rc = _lib.load().qb_vi_sample(qb_dtype(dt), _ptr(mu), _ptr(rho), _ptr(eps), nsam, P, float(pi), float(sigma1),
                                      float(sigma2), use_seed, int(step), _ptr(w), _ptr(logq), _ptr(logp), _stream())
    _lib.check(rc, 'qb_vi_sample')
    return w, eps, logq, logp


def vi_backward(mu, rho, eps, w, glp, pi, sigma1, sigma2, c_ssq, c_logp, c_logq):
    nsam, P = w.shape
    gmu = torch.empty_like(mu)
    grho = torch.empty_like(rho)
    with torch.cuda.device(mu.device):
        rc = _lib.load().qb_vi_backward(qb_dtype(mu.dtype), _ptr(mu), _ptr(rho), _ptr(eps), _ptr(w), _ptr(glp), nsam, P,
                                        float(pi), float(sigma1), float(sigma2), float(c_ssq), float(c_logp),
                                        float(c_logq), _ptr(gmu), _ptr(grho), _stream())
    _lib.check(rc, 'qb_vi_backward')
    return gmu, grho


def fma_peak(dtype=torch.float32, variant=0, iters=20000, device='cuda', repeats=5):
    """Measured FMA throughput (FLOP/s) of the CUDA cores: the roofline denominator for kernels 1-4."""
    dev = torch.device(device)
    sink = torch.zeros(4, dtype=dtype, device=dev)
    flops = C.c_double(0.0)
    lib = _lib.load()
    best = 0.0
    with torch.cuda.device(dev):
        for _ in range(repeats + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.qb_fma_peak(qb_dtype(dtype), variant, iters, C.byref(flops), _ptr(sink), _stream()), 'qb_fma_peak')
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1)
            best = max(best, flops.value / (ms * 1e-3))
    return best
