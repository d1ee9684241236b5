"""NNWrap: the numpy <-> network seam of the reference (quinn/nns/nnwrap.py:9-150, 330-347), backed by
the CUDA kernels: ``__call__`` / ``predict`` / ``nn_p`` run posterior-predictive kernel 4,
``calc_loss`` / ``calc_lossgrad`` with a NegLogPost run kernels 1 / 2, ``calc_hess_full`` kernel 5, ``kfac_device``
kernel 6.  No torch-CPU evaluation."""
import numpy as np
import torch

from .. import ops
from ..netdesc import netdesc_from_module
from .losses import NegLogPost
from .tchutils import tch

_DEFAULT_DEVICE = 'cuda'


def _dtype_of(module):
    for p in module.parameters():
        return p.dtype if p.dtype in (torch.float32, torch.float64) else torch.float64
    return torch.float64


def device_forward(module, x, theta=None, dtype=None):
    """module(x) evaluated by kernel 4 at flat parameters `theta` (default: the module's own)."""
    desc = netdesc_from_module(module)
    dtype = dtype or _dtype_of(module)
    if theta is None:
        theta = torch.cat([p.detach().flatten() for p in module.parameters()])
    out, _, _ = ops.predict(desc, theta, np.asarray(x) if not torch.is_tensor(x) else x, dtype=dtype,
                            device=_DEFAULT_DEVICE)
    return out[0].double().cpu().numpy() if dtype == torch.float64 else out[0].cpu().numpy()


class NNWrap:
    def __init__(self, nnmodel):
        self.nnmodel = nnmodel
        self.indices = None
        self._desc = None
        self._prob_key = None
        self._prob = None
        self.p_flatten()

    # ---- flat layout (nnwrap.py:64-106)
    def p_flatten(self):
        flats = [torch.flatten(p) for p in self.nnmodel.parameters()]
        self.indices, s = [], 0
        for f in flats:
            self.indices.append((s, s + f.shape[0]))
            s += f.shape[0]
        return torch.cat(flats).view(-1, 1)

    def p_unflatten(self, flat_parameter):
        """Fill the module's parameters from a flat numpy vector; returns the list of tensors."""
        device = getattr(self.nnmodel, 'device', 'cpu')
        out = []
        for (s, e), p in zip(self.indices, self.nnmodel.parameters()):
            t = tch(np.asarray(flat_parameter[s:e]), device=device).to(p.dtype)
            if p.dim() > 0:
                t = t.view(*p.shape)
            p.data = t
            out.append(t)
        return out

    def desc(self):
        if self._desc is None:
            self._desc = netdesc_from_module(self.nnmodel)
        return self._desc

    # ---- evaluation
    def __call__(self, x):
        return device_forward(self.nnmodel, x)

    def predict(self, x_in, weights):
        self.p_unflatten(weights)
        return device_forward(self.nnmodel, x_in, theta=np.asarray(weights))

    def _problem(self, loss_fn, inputs, targets):
        if not isinstance(loss_fn, NegLogPost):
            raise NotImplementedError(
                'quinn_b200.NNWrap evaluates losses in fused CUDA kernels and only knows NegLogPost '
                '(the loss every sampler uses, SURVEY.md section 2 row 3); other loss modules have no GPU path here')
        inputs, targets = np.asarray(inputs, dtype=np.float64), np.asarray(targets, dtype=np.float64)
        # content key: data bytes, likelihood and prior values (equal-shape / equal-sum data no longer collide, in-place
        # edits of the loss module or of the anchor are seen)
        import hashlib
        hsh = hashlib.blake2b(np.ascontiguousarray(inputs).tobytes(), digest_size=16)
        hsh.update(np.ascontiguousarray(targets).tobytes())
        pp0 = loss_fn.priorparams
        if pp0 is not None:
            hsh.update(np.ascontiguousarray(np.asarray(pp0['anchor'].detach().cpu() if hasattr(pp0['anchor'], 'detach') else pp0['anchor'],
                                                       dtype=np.float64)).tobytes())
        key = (inputs.shape, targets.shape, hsh.hexdigest(), float(loss_fn.sigma), loss_fn.fulldatasize,
               None if pp0 is None else float(pp0['sigma']))
        if key != self._prob_key:
            pp = loss_fn.priorparams
            self._prob = ops.Problem(self.desc(), inputs, targets, float(loss_fn.sigma), dtype=_dtype_of(self.nnmodel),
                                     device=_DEFAULT_DEVICE,
                                     prior_sigma=None if pp is None else float(pp['sigma']),
                                     prior_anchor=None if pp is None else pp['anchor'],
                                     fulldatasize=loss_fn.fulldatasize)
            self._prob_key = key
        return self._prob

    def calc_loss(self, weights, loss_fn, inputs, targets):
        """loss(theta) as a Python float (nnwrap.py:109-126); NegLogPost -> kernel 1."""
        prob = self._problem(loss_fn, inputs, targets)
        self.p_unflatten(weights)          # the reference leaves the model at `weights` too
        return float(-ops.logpost(prob, np.asarray(weights, dtype=np.float64))[0].item())

    def calc_lossgrad(self, weights, loss_fn, inputs, targets):
        """d loss / d theta as a flat numpy vector (nnwrap.py:128-150); NegLogPost -> kernel 2."""
        prob = self._problem(loss_fn, inputs, targets)
        self.p_unflatten(weights)
        _, g = ops.logpost_grad(prob, np.asarray(weights, dtype=np.float64))
        return -g[0].double().cpu().numpy()


    # ---- diagonal Fisher (the by-product of kernel 2 that NN_Laplace uses, SURVEY.md 8f rank 4)
    def calc_fisher_diag(self, weights, loss_fn, inputs, targets, chunk=65536):
        """Diagonal of calc_hess_diag as a numpy vector (fisher_diag_device)."""
        return self.fisher_diag_device(weights, loss_fn, inputs, targets, chunk).cpu().numpy()

    def fisher_diag_device(self, weights, loss_fn, inputs, targets, chunk=65536):
        """Diagonal of calc_hess_diag as a float64 device vector: mean over the data points of the squared gradient of the
        loss evaluated on one point at a time (nnwrap.py:204-229).  Kernel 2 runs with one data point per "member"
        (qb_logpost_members: member i sees x[i], y[i]; all members share theta), qb_colsq_mean reduces the squares."""
        import ctypes as C
        from .. import _lib, post
        from ..ops import _ptr, _stream
        prob = self._problem(loss_fn, inputs, targets)
        self.p_unflatten(weights)
        N, P, o = prob.n, prob.desc.n_params, prob.desc.out_dim
        theta = prob.theta(np.asarray(weights, dtype=np.float64))
        lik = _lib.qb_lik_t(prob.clik.sigma, prob.clik.prior_sigma, 0.0, prob.clik.prior_anchor, 0, 0)
        if loss_fn.priorparams is not None:
            lik.prior_scale = float(o) / float(loss_fn.fulldatasize)      # a single point: len(predictions) == o (losses.py:199-204)
        lib = _lib.load()
        acc = torch.zeros(P, dtype=torch.float64, device=prob.device)
        for lo in range(0, N, chunk):
            n = min(chunk, N - lo)
            th = theta.expand(n, P).contiguous()
            lp = torch.empty(n, dtype=torch.float64, device=prob.device)
            g = torch.empty((n, P), dtype=prob.dtype, device=prob.device)
            need = lib.qb_eval_workspace_bytes(C.byref(prob.cnet), prob.qdt, n, 1, 1)
            ws = torch.empty(max(int(need), 256), dtype=torch.uint8, device=prob.device)
            data = _lib.qb_data_t(prob.x[lo:lo + n].data_ptr(), prob.y[lo:lo + n].data_ptr(), 1)
            with torch.cuda.device(prob.device):
                _lib.check(lib.qb_logpost_members(C.byref(prob.cnet), prob.qdt, _ptr(th), n, C.byref(data), prob.desc.in_dim, o,
                                                  C.byref(lik), _ptr(lp), _ptr(g), _ptr(ws), ws.numel(), _stream()),
                           'qb_logpost_members')
            acc += post.fisher_diag(g) * (n / float(N))
        return acc

    def hess_full_device(self, weights, loss_fn, inputs, targets):
        """Hessian of the loss (= -d^2 lp / d theta^2) as a (P, P) device tensor: P exact Hessian-vector products of
        unit directions in kernel 5."""
        prob = self._problem(loss_fn, inputs, targets)
        self.p_unflatten(weights)
        return ops.logpost_hessian(prob, np.asarray(weights, dtype=np.float64)).neg_()

    def calc_hess_full(self, weights, loss_fn, inputs, targets):
        """(P, P) Hessian of the loss as numpy (nnwrap.py:153-203); NegLogPost -> kernel 5."""
        return self.hess_full_device(weights, loss_fn, inputs, targets).double().cpu().numpy()

    def kfac_device(self, weights, loss_fn, inputs, targets):
        """Kronecker factors of the per-point empirical Fisher of every Linear layer (kernel 6): a list of dicts
        {A, s, G} of float64 device tensors, raw sums over the data points (ops.logpost_kfac)."""
        prob = self._problem(loss_fn, inputs, targets)
        self.p_unflatten(weights)
        return ops.logpost_kfac(prob, np.asarray(weights, dtype=np.float64))

    def calc_hess_diag(self, weights, loss_fn, inputs, targets):
        """The reference's return value: a (P, P) matrix with the diagonal Fisher on its diagonal (nnwrap.py:229)."""
        return np.diag(self.calc_fisher_diag(weights, loss_fn, inputs, targets))


def nnwrapper(x, nnmodel):
    return device_forward(nnmodel, x)


def nn_p(p, x, *otherpars):
    """NN_p(x) for a flat parameter vector p (nnwrap.py:330-347)."""
    nnw = NNWrap(otherpars[0])
    return nnw.predict(x, p)
