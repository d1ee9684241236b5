from .quinn import QUiNNBase
from .nn_mcmc import NN_MCMC
from .nn_ens import NN_Ens
from .nn_rms import NN_RMS
from .nn_vi import NN_VI
from .nn_laplace import NN_Laplace
