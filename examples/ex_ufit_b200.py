#!/usr/bin/env python
"""The reference's examples/ex_ufit.py workflow (methods amcmc / hmc / ens / vi / laplace) with quinn_b200 as a drop-in:
only the imports change.  Plotting is out of scope, so the script prints predictive moments instead.

    python examples/ex_ufit_b200.py amcmc|hmc|ens|vi|laplace [nchains]
"""
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from quinn_b200.solvers import NN_MCMC, NN_Ens, NN_VI, NN_Laplace      # noqa: E402  (reference: from quinn.solvers.nn_mcmc import NN_MCMC ...)
from quinn_b200.nns import RNet, Poly                      # noqa: E402  (reference: from quinn.nns.rnet import RNet, Poly)


def main():
    meth = sys.argv[1] if len(sys.argv) > 1 else 'amcmc'
    nchains = int(sys.argv[2]) if len(sys.argv) > 2 else None
    np.random.seed(0)
    torch.manual_seed(0)
    nall, ndim, datanoise = 15, 1, 0.02
    xall = np.random.rand(nall, ndim) * 2 * np.pi - np.pi                       # scale01ToDom(rand, [-pi, pi])
    yall = datanoise * np.random.randn(nall, 1) + np.sum(np.sin(xall), axis=1).reshape(-1, 1)   # Sine
    ntrn = int(0.9 * nall)
    xtrn, ytrn, xval, yval = xall[:ntrn], yall[:ntrn], xall[ntrn:], yall[ntrn:]
    nnet = RNet(3, 3, wp_function=Poly(0), indim=ndim, outdim=1, layer_pre=True, layer_post=True,
                biasorno=True, nonlin=True, mlp=False, final_layer=None)
    if meth == 'amcmc':
        uqnet = NN_MCMC(nnet, verbose=True)
        uqnet.fit(xtrn, ytrn, zflag=False, datanoise=datanoise, nmcmc=10000, sampler='amcmc', sampler_params={'gamma': 0.01},
                  nchains=nchains)
    elif meth == 'hmc':
        uqnet = NN_MCMC(nnet, verbose=True)
        uqnet.fit(xtrn, ytrn, zflag=False, datanoise=datanoise, nmcmc=10000, sampler='hmc',
                  sampler_params={'L': 3, 'epsilon': 0.0025}, nchains=nchains)
    elif meth == 'vi':
        uqnet = NN_VI(nnet, verbose=True)
        uqnet.fit(xtrn, ytrn, val=[xval, yval], datanoise=datanoise, lrate=0.01, batch_size=None, nsam=1, nepochs=2000)
    elif meth == 'ens':
        uqnet = NN_Ens(nnet, nens=3, dfrac=0.8, verbose=True)
        uqnet.fit(xtrn, ytrn, val=[xval, yval], lrate=0.01, batch_size=2, nepochs=300)
    elif meth == 'laplace':
        uqnet = NN_Laplace(nnet, nens=3, la_type='full', cov_scale=1.0, datanoise=datanoise, priorsigma=1.0, dfrac=0.8,
                           verbose=True)
        uqnet.fit(xtrn, ytrn, val=[xval, yval], lrate=0.01, batch_size=2, nepochs=300)
    else:
        raise SystemExit('pick among amcmc, hmc, vi, ens, laplace')
    xgrid = np.linspace(-np.pi, np.pi, 11)[:, None]
    nsam = 3 if meth == 'ens' else 1000
    mean, var, _ = uqnet.predict_mom_sample(xgrid, msc=1, nsam=nsam)
    print('x        truth    mean     std')
    for xg, m, v in zip(xgrid[:, 0], mean[:, 0], var[:, 0]):
        print(f'{xg:8.3f} {np.sin(xg):8.3f} {m:8.3f} {np.sqrt(max(v, 0)):8.3f}')


if __name__ == '__main__':
    main()
