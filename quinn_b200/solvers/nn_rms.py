"""NN_RMS: randomised-MAP-sampling ensemble with the reference's interface (quinn/solvers/nn_rms.py:10-56; Pearce et al.
2018).  Every member minimises NegLogPost (losses.py:186-206) with its own random prior anchor; with the default Adam
options all members are trained TOGETHER on the device (quinn_b200/ens/batched.py: kernels 1 / 2 evaluate the
anchored log-posterior of member k through `anchor_per_chain`), other nnfit options keep the member-by-member loop."""
import copy

import numpy as np
import torch

from ..netdesc import netdesc_from_module, flatten_module, unflatten_module
from .nn_ens import NN_Ens


class NN_RMS(NN_Ens):
    def __init__(self, nnmodel, datanoise=0.1, priorsigma=1.0, **kwargs):
        super().__init__(nnmodel, **kwargs)
        self.datanoise = datanoise
        self.priorsigma = priorsigma
        self.nparams = sum(p.numel() for p in self.nnmodel.parameters())

    def fit(self, xtrn, ytrn, **kwargs):
        """Same call as the reference (nn_rms.py:33-56): per member a random subset (np.random.permutation), an anchor
        torch.randn(P) * priorsigma and nnfit(loss_fn='logpost', datanoise, priorparams).  The members' subsets and
        anchors are kept as `subsets` [nens, nsub] and `anchors` [nens, P]."""
        ntrn = ytrn.shape[0]
        nsub = int(ntrn * self.dfrac)
        user = dict(kwargs)
        for k in ('loss_fn', 'datanoise', 'priorparams'):
            user.pop(k, None)
        self.batched_fit = False
        if not self._can_batch(user):
            subsets, anchors = [], []
            for jens, learner in enumerate(self.learners):
                print(f"======== Fitting Learner {jens + 1}/{self.nens} =======")
                ind = np.random.permutation(ntrn)[:nsub]
                anchor = torch.randn(size=(self.nparams,), dtype=torch.float64) * self.priorsigma
                kw = dict(user, lhist_suffix=f'_e{jens}', loss_fn='logpost', datanoise=self.datanoise,
                          priorparams={'sigma': self.priorsigma, 'anchor': anchor})
                learner.fit(xtrn[ind], ytrn[ind], **kw)
                subsets.append(ind)
                anchors.append(anchor.numpy())
            self.subsets, self.anchors = np.stack(subsets), np.stack(anchors)
            return
        from ..ens.batched import fit_members
        print(f"======== Fitting {self.nens} anchored learners together =======")
        nepochs = user.get('nepochs', 5000)
        bs = user.get('batch_size')
        subsets, anchors, perms = [], [], []
        for _ in range(self.nens):
            # the reference's order of random draws: subset, anchor, then one torch.randperm per epoch inside nnfit
            # (nnfit.py:126, also when the batch is the whole subset)
            subsets.append(np.random.permutation(ntrn)[:nsub])
            anchors.append((torch.randn(size=(self.nparams,), dtype=torch.float64) * self.priorsigma).numpy())
            perms.append(np.stack([torch.randperm(nsub).numpy() for _ in range(nepochs)]) if nepochs * nsub <= 5 * 10 ** 7 else None)
        use_perms = bs is not None and bs < nsub and all(p is not None for p in perms)
        desc = netdesc_from_module(self.learners[0].nnmodel)
        theta0 = np.stack([flatten_module(l.nnmodel) for l in self.learners])
        res = fit_members(desc, theta0, np.asarray(xtrn), np.asarray(ytrn), np.stack(subsets), val=user.get('val'),
                          nepochs=nepochs, lrate=user.get('lrate', 0.1), wd=user.get('wd', 0.0), batch_size=bs,
                          perms=np.stack(perms) if use_perms else None, dtype=self.dtype, freq_out=user.get('freq_out', 100),
                          logpost=dict(sigma=self.datanoise, prior_sigma=self.priorsigma, anchor=np.stack(anchors)))
        best = res['best_theta'].double().cpu().numpy()
        self.fit_info = {k: v.cpu().numpy() for k, v in res.items() if k in ('best_loss', 'best_epoch')}
        self.subsets, self.anchors = np.stack(subsets), np.stack(anchors)
        self.batched_fit = True
        for k, learner in enumerate(self.learners):
            learner.best_model = copy.deepcopy(learner.nnmodel)
            unflatten_module(learner.best_model, best[k])
            learner.trained = True
