"""NN_Laplace: Laplace approximation around anchored MAP fits (quinn/solvers/nn_laplace.py:76-139, SURVEY.md row 18).

Every member is fitted exactly as NN_RMS fits it (same random draws, same batched / member-by-member choice); then the
curvature of its NegLogPost at the MAP is taken on the device, either the exact Hessian (la_type='full': kernel 5, one
Hessian-vector product per unit direction), the diagonal Fisher of NNWrap.calc_hess_diag (la_type='diag') or the
Kronecker-factored Fisher of every Linear layer (la_type='kron': kernel 6, DESIGN.md section 4g).  The curvature is
factored on the device (torch.linalg.eigh, elementwise, or eigh of each layer's two factors) and the posterior draws
theta = mu_j + H_j^{-1/2} z sqrt(cov_scale) are formed there, so predictions go straight to kernel 4.  predict_mom_glm is
the linearised predictive instead: per-point Jacobians from kernel 7 (DESIGN.md section 4h) contracted with the same
covariance, no sampling."""
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

    def predict_mom_glm(self, x, msc=0):
        """Moments of the linearised (GLM) predictive f(x; mu_j) + J_j(x) (theta - mu_j), theta ~ N(mu_j, cov_scale
        Sigma_j), with Sigma_j the covariance _ens_thetas samples from; members weigh equally.  Deterministic, no
        observation noise.  Same contract as predict_mom_sample: (mean [N, o], var [N, o] for msc >= 1, cov [N, N, o]
        for msc == 2), numpy float64.  J_j comes from kernel 7 in the solver's dtype; the contraction with Sigma_j runs
        in float64 on the device, over chunks of points whose buffers stay under _GLM_CHUNK_BYTES each."""
        if msc not in (0, 1, 2):
            raise ValueError(f"msc={msc}, but needs to be 0,1, or 2.")
        if self.means is None:
            raise RuntimeError('predict_mom_glm needs the posterior: call fit first')
        from .. import ops
        desc = self._desc()
        x = np.asarray(x)
        N, o, P = x.shape[0], desc.out_dim, desc.n_params
        dev = self.means.device
        F = ops.jac_plan_info(desc, max(N, 1), self.dtype)['rows']
        step = max(1, _GLM_CHUNK_BYTES // (8 * max(F, o * P)))
        vsum = torch.zeros((N, o), dtype=torch.float64, device=dev)
        csum = torch.zeros((o, N, N), dtype=torch.float64, device=dev) if msc == 2 else None
        fmem = torch.zeros((self.nens, N, o), dtype=torch.float64, device=dev)
        for j in range(self.nens):
            mu = self.means[j].to(self.dtype)
            Bs = []
            for lo in range(0, N, step):
                f, pairs = ops.predict_jac(desc, mu, x[lo:lo + step], dtype=self.dtype, device=dev)
                fmem[j, lo:lo + step] = f
                if msc == 2:
                    Bs.append(_glm_factor(self.la_type, self._factors[j], desc, pairs))
                elif msc == 1:
                    vsum[lo:lo + step] += _glm_var(self.la_type, self._factors[j], desc, pairs)
            if msc == 2 and Bs:
                B = torch.cat(Bs)
                csum += torch.einsum('nja,mja->jnm', B, B)
        # law of total variance over equally weighted members, as the mean of the members' variances plus the variance of
        # their means (the same value as mean_j(v_j + f_j^2) - mean^2, without its cancellation)
        mean = fmem.mean(0)
        dev_f = fmem - mean
        var = cov = None
        if msc == 2:
            cv = self.cov_scale * csum / self.nens + torch.einsum('knj,kmj->jnm', dev_f, dev_f) / self.nens  # [o, N, N]
            var = torch.diagonal(cv, dim1=1, dim2=2).T.cpu().numpy()
            cov = cv.permute(1, 2, 0).cpu().numpy()
        elif msc == 1:
            var = (self.cov_scale * vsum / self.nens + (dev_f * dev_f).mean(0)).cpu().numpy()
        return mean.cpu().numpy(), var, cov


_GLM_CHUNK_BYTES = 1 << 30        # predict_mom_glm: the largest buffer of one chunk of points


def assemble_jac(desc, pairs):
    """J [n, o, P] (float64) of d f_j(x_n) / d theta from kernel 7's per-layer pairs (ops.predict_jac): layer l adds
    coef_m * outer(d_l[j, :, n], [a_l[:, n]; 1]) at each of its terms (coef_m, w_off_m, b_off_m), so layers that share
    weights sum their parts.  Runs wherever the pair tensors live."""
    a0 = pairs[0]['a']
    n, o = a0.shape[1], desc.out_dim
    J = torch.zeros((n, o, desc.n_params), dtype=torch.float64, device=a0.device)
    for L, p in zip(desc.layers, pairs):
        a, d = p['a'].double(), p['d'].double()
        gW = torch.einsum('jun,in->njui', d, a).reshape(n, o, L.n_out * L.n_in)
        gb = d.permute(2, 0, 1)
        for c, wo, bo in (L.terms or [(1.0, L.w_off, L.b_off)]):
            J[:, :, wo:wo + L.n_out * L.n_in] += c * gW
            if bo >= 0:
                J[:, :, bo:bo + L.n_out] += c * gb
    return J


def _glm_factor(la_type, fac, desc, pairs):
    """B [n, o, K] with B[n, j] B[m, j]^T = J_j(x_n) Sigma J_j(x_m)^T for one member's factors"""
    if la_type == 'full':
        U, isq, _ = fac
        return assemble_jac(desc, pairs) @ (U * isq)
    if la_type == 'diag':
        return assemble_jac(desc, pairs) * fac[0]
    Bs = []
    for p, (_, UG, UA, isq, _) in zip(pairs, fac):
        dr, ar = _kron_rotate(p, UG, UA)                     # [o, n_out, n], [n_in(+1), n]
        B = dr.permute(2, 0, 1)[:, :, :, None] * ar.T[:, None, None, :] * isq
        Bs.append(B.reshape(B.shape[0], B.shape[1], -1))
    return torch.cat(Bs, 2)


def _glm_var(la_type, fac, desc, pairs):
    """diag of J Sigma J^T [n, o] for one member's factors ('kron': per layer sum_rc d'_r^2 a'_c^2 / lambda_rc, with
    d' = U_G^T d and a' = U_A^T [a; 1], no assembly)"""
    if la_type != 'kron':
        return (_glm_factor(la_type, fac, desc, pairs) ** 2).sum(2)
    v = 0.0
    for p, (_, UG, UA, isq, _) in zip(pairs, fac):
        dr, ar = _kron_rotate(p, UG, UA)
        M = (isq * isq) @ (ar * ar)                          # [n_out, n]: sum_c a'_c^2 / lambda_rc
        v = v + ((dr * dr) * M[None]).sum(1).T
    return v


def _kron_rotate(p, UG, UA):
    a, d = p['a'].double(), p['d'].double()
    if UA.shape[0] > a.shape[0]:                             # a layer with a bias: a~ = [a; 1]
        a = torch.cat([a, torch.ones((1, a.shape[1]), dtype=a.dtype, device=a.device)])
    return torch.einsum('ur,jun->jrn', UG, d), UA.T @ a


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
