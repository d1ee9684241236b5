from .mcmc import MCMCBase, DeviceLogPost
from .admcmc import AMCMC
from .hmc import HMC
from .mala import MALA
from .nuts import NUTS
from .pt import PT
