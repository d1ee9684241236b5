"""NN_Laplace: Laplace approximation around anchored MAP fits (quinn/solvers/nn_laplace.py:76-139, SURVEY.md row 18).

Every member is fitted exactly as NN_RMS fits it (same random draws, same batched / member-by-member choice); then the
curvature of its NegLogPost at the MAP is taken on the device, either the exact Hessian (la_type='full': kernel 5, one
Hessian-vector product per unit direction) or the diagonal Fisher of NNWrap.calc_hess_diag (la_type='diag').  The
curvature is factored on the device (torch.linalg.eigh, or elementwise) and the posterior draws
theta = mu_j + H_j^{-1/2} z sqrt(cov_scale) are formed there, so predictions go straight to kernel 4."""
import copy
import warnings

import numpy as np
import torch

from ..netdesc import flatten_module
from ..nns.losses import NegLogPost
from ..nns.nnwrap import NNWrap
from .nn_rms import NN_RMS


class NN_Laplace(NN_RMS):
    def __init__(self, nnmodel, nens=1, la_type='full', cov_scale=1.0, datanoise=0.1, priorsigma=1.0, dfrac=1.0,
                 verbose=False, dtype=torch.float64):
        if la_type not in ('full', 'diag'):
            raise ValueError(f"la_type={la_type!r}, but needs to be 'full' or 'diag'")
        super().__init__(nnmodel, datanoise=datanoise, priorsigma=priorsigma, nens=nens, dfrac=dfrac, verbose=verbose,
                         dtype=dtype)
        self.la_type = la_type
        self.cov_scale = cov_scale
        self.means = None         # [nens, P] device tensor: the members' MAP parameters
        self._factors = []        # per member: (U, |lambda|^-1/2, lambda) for 'full', (F^-1/2, F) for 'diag'
        self._cov_mats = None

    def fit(self, xtrn, ytrn, **kwargs):
        """NN_RMS.fit, then la_calc on every member's best model with the member's data subset and anchor."""
        super().fit(xtrn, ytrn, **kwargs)
        self._factors, self._cov_mats = [], None
        means = [self.la_calc(learner, xtrn[self.subsets[k]], ytrn[self.subsets[k]], self.anchors[k])
                 for k, learner in enumerate(self.learners)]
        self.means = torch.stack(means)

    def la_calc(self, learner, xtrn, ytrn, anchor):
        """Curvature of NegLogPost(model, nsub, datanoise, {'sigma': priorsigma, 'anchor': anchor}) at the member's MAP,
        factored on the device.  Returns the MAP as a device tensor."""
        model = copy.deepcopy(learner.best_model).to(self.dtype)       # the curvature is taken in the solver's dtype
        theta = flatten_module(model)
        loss = NegLogPost(model, xtrn.shape[0], self.datanoise,
                          {'sigma': self.priorsigma, 'anchor': torch.as_tensor(anchor, dtype=torch.float64)})
        nnw = NNWrap(model)
        if self.la_type == 'full':
            H = nnw.hess_full_device(theta, loss, xtrn, ytrn).double()
            H = 0.5 * (H + H.T)            # exact up to rounding; eigh reads one triangle
            lam, U = torch.linalg.eigh(H)
            if bool((lam == 0).any()):
                raise np.linalg.LinAlgError('Singular matrix')
            if bool((lam < 0).any()):
                # numpy's multivariate_normal factors the covariance by SVD and samples with |lambda|
                warnings.warn('covariance is not symmetric positive-semidefinite.', RuntimeWarning, stacklevel=2)
            self._factors.append((U, lam.abs().rsqrt(), lam))
            dev = H.device
        else:
            F = nnw.fisher_diag_device(theta, loss, xtrn, ytrn)
            if bool((F == 0).any()):
                raise np.linalg.LinAlgError('Singular matrix')
            self._factors.append((F.rsqrt(), F))
            dev = F.device
        return torch.as_tensor(theta, dtype=torch.float64, device=dev)      # on the device the curvature lives on

    @property
    def cov_mats(self):
        """Host list of the members' covariances H^-1 without cov_scale (what the reference keeps), built on first use."""
        if self._cov_mats is None:
            mats = []
            for f in self._factors:
                if self.la_type == 'full':
                    U, _, lam = f
                    mats.append(((U / lam) @ U.T).cpu().numpy())
                else:
                    mats.append(np.diag((1.0 / f[1]).cpu().numpy()))
            self._cov_mats = mats
        return self._cov_mats

    def _ens_thetas(self, nsam):
        """nsam posterior draws: member indices from np.random.randint, standard normals drawn on the device from a seed
        taken from np.random (np.random.seed makes them repeatable)."""
        members = np.random.randint(0, self.nens, size=nsam)
        seed = int(np.random.randint(0, 2 ** 31 - 1))
        dev = self.means.device
        gen = torch.Generator(device=dev)
        gen.manual_seed(seed)
        z = torch.randn((nsam, self.means.shape[1]), generator=gen, dtype=torch.float64, device=dev)
        thetas = torch.empty_like(z)
        sc = float(np.sqrt(self.cov_scale))
        for j in np.unique(members):
            rows = torch.as_tensor(np.nonzero(members == j)[0], device=dev)
            if self.la_type == 'full':
                U, isq, _ = self._factors[j]
                thetas[rows] = self.means[j] + ((z[rows] * isq) @ U.T) * sc
            else:
                isq, _ = self._factors[j]
                thetas[rows] = self.means[j] + z[rows] * isq * sc
        return self._desc(), thetas.to(self.dtype), self.dtype

    def predict_sample(self, x):
        """One draw theta ~ N(mu_j, cov_scale H_j^-1) of a random member, evaluated by kernel 4."""
        from .. import ops
        desc, thetas, dtype = self._ens_thetas(1)
        out, _, _ = ops.predict(desc, thetas, np.asarray(x), dtype=dtype)
        return out[0].double().cpu().numpy()
