"""NN_Laplace: Laplace approximation around anchored MAP fits (quinn/solvers/nn_laplace.py:76-139, SURVEY.md row 18).

Every member is fitted exactly as NN_RMS fits it (same random draws, same batched / member-by-member choice); then the
curvature of its NegLogPost at the MAP is taken on the device, either the exact Hessian (la_type='full': kernel 5, one
Hessian-vector product per unit direction), the diagonal Fisher of NNWrap.calc_hess_diag (la_type='diag') or the
Kronecker-factored Fisher of every Linear layer (la_type='kron': kernel 6, DESIGN.md section 4g).  The curvature is
factored on the device (torch.linalg.eigh, elementwise, or eigh of each layer's two factors) and the posterior draws
theta = mu_j + H_j^{-1/2} z sqrt(cov_scale) are formed there, so predictions go straight to kernel 4."""
import copy
import warnings

import numpy as np
import torch

from ..netdesc import flatten_module, netdesc_from_module
from ..nns.losses import NegLogPost
from ..nns.nnwrap import NNWrap
from .nn_rms import NN_RMS


class NN_Laplace(NN_RMS):
    def __init__(self, nnmodel, nens=1, la_type='full', cov_scale=1.0, datanoise=0.1, priorsigma=1.0, dfrac=1.0,
                 verbose=False, dtype=torch.float64):
        if la_type not in ('full', 'diag', 'kron'):
            raise ValueError(f"la_type={la_type!r}, but needs to be 'full', 'diag' or 'kron'")
        if la_type == 'kron':
            _check_kron_net(netdesc_from_module(nnmodel))
        super().__init__(nnmodel, datanoise=datanoise, priorsigma=priorsigma, nens=nens, dfrac=dfrac, verbose=verbose,
                         dtype=dtype)
        self.la_type = la_type
        self.cov_scale = cov_scale
        self.means = None         # [nens, P] device tensor: the members' MAP parameters
        # per member: (U, |lambda|^-1/2, lambda) for 'full', (F^-1/2, F) for 'diag', and for 'kron' a list of per-layer
        # (theta index [n_out, n_in(+1)], U_G, U_A, lambda^-1/2, lambda)
        self._factors = []
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
        elif self.la_type == 'kron':
            facs = nnw.kfac_device(theta, loss, xtrn, ytrn)
            # the per-point prior share o / fulldatasize of 'diag' (oracle diag_fisher), as a Hessian: tau I
            tau = (np.shape(ytrn)[1] / loss.fulldatasize) / float(self.priorsigma) ** 2
            self._factors.append(_kron_factors(nnw.desc(), facs, xtrn.shape[0], tau))
            dev = facs[0]['A'].device
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
                elif self.la_type == 'kron':
                    cov = np.zeros((self.nparams, self.nparams))
                    for idx, UG, UA, _, lam in f:
                        Q = torch.kron(UG, UA)                   # (j, i) row-major, as idx
                        ii = idx.reshape(-1).cpu().numpy()
                        cov[np.ix_(ii, ii)] = ((Q / lam.reshape(-1)) @ Q.T).cpu().numpy()
                    mats.append(cov)
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
            elif self.la_type == 'kron':
                th = self.means[j].expand(len(rows), -1).clone()
                zr = z[rows]
                for idx, UG, UA, isq, _ in self._factors[j]:
                    E = UG @ (zr[:, idx] * isq) @ UA.T                  # [n, n_out, n_in(+1)]: Lambda_l^-1/2 z
                    th[:, idx] += E * sc
                thetas[rows] = th
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


def _check_kron_net(desc):
    """'kron' needs every Linear layer to own its weights: no shared (RNet Poly(0)) or polynomial-in-depth weights."""
    seen = set()
    for L in desc.layers:
        if L.terms and len(L.terms) > 1:
            raise ValueError("la_type='kron' needs a network whose layers own their weights: polynomial-in-depth "
                             "weights (RNet with Lin / Quad / Cubic / Poly(n)) are not supported")
        if L.w_off in seen:
            raise ValueError("la_type='kron' needs a network whose layers own their weights: shared weights (RNet with "
                             "Poly(0)) are not supported")
        seen.add(L.w_off)


def _kron_factors(desc, facs, n, tau):
    """Per layer (theta index, U_G, U_A, lambda^-1/2, lambda) of Lambda_l = G/n (x) A~/n + tau I, eigenvalues
    lambda[j, i] = g_j a_i + tau; the factors are PSD by construction, so negative eigenvalues are rounding (set to 0)."""
    out = []
    for L, f in zip(desc.layers, facs):
        A, G = f['A'], f['G']
        dev = A.device
        if f['s'] is not None:
            nn = torch.full((1, 1), float(n), dtype=A.dtype, device=dev)
            A = torch.cat([torch.cat([A, f['s'][:, None]], 1), torch.cat([f['s'][None, :], nn], 1)], 0)
        la, UA = torch.linalg.eigh(A / n)
        lg, UG = torch.linalg.eigh(G / n)
        lam = lg.clamp(min=0.0)[:, None] * la.clamp(min=0.0)[None, :] + tau
        if bool((lam == 0).any()):
            raise np.linalg.LinAlgError('Singular matrix')
        idx = L.w_off + torch.arange(L.n_out, device=dev)[:, None] * L.n_in + torch.arange(L.n_in, device=dev)[None, :]
        if L.b_off >= 0:
            idx = torch.cat([idx, (L.b_off + torch.arange(L.n_out, device=dev))[:, None]], 1)
        out.append((idx, UG, UA, lam.rsqrt(), lam))
    covered = torch.zeros(desc.n_params, dtype=torch.bool, device=out[0][0].device)
    for idx, *_ in out:
        covered[idx.reshape(-1)] = True
    if not bool(covered.all()):
        raise ValueError("la_type='kron' needs every parameter to belong to one Linear layer")
    return out
