"""Hot-path distributions, plus the two location-scale families of SURVEY 8(f)-4 (Logistic, Laplace) on the same
kernel templates.  and Uniform, Poisson for count data and Beta for probabilities.  The reference's remaining wrappers
over torch.distributions (gamma, studentT, exponential; zhusuan/distributions/__init__.py:3-13) are outside the
accelerated path and are not rebuilt here (SURVEY.md §2 #5, DESIGN.md §scope)."""
from .base import *
from .normal import *
from .bernoulli import *
from .categorical import *
from .logistic import *
from .laplace import *
from .uniform import *
from .poisson import *
from .beta import *

# Latent nodes draw their sample and its log q in one launch when the node's event reduction allows it
# (zs_normal_latent_fwd / zs_bernoulli_latent_fwd); set to False to always use the separate kernels.
FUSED_LATENT = True
