"""lsqfitgp_b200: B200-native (sm_100a) implementation of lsqfitgp's GP-fitting hot path.

Drop-in for the path Gram build -> Cholesky -> solves / log-determinant behind the lsqfitgp API
(`GP`, kernels, `_linalg.Chol`, `empbayes_fit`); see DESIGN.md for the scope and INTEGRATION.md for the
C ABI.  Public names follow src/lsqfitgp/__init__.py:32-70 of the reference, restricted to the path.
"""

__version__ = '0.1.0'

from . import _lib  # noqa: F401
from ._array import StructuredArray, unstructured_to_structured, asarray
from ._Deriv import Deriv
from ._Kernel import (CrossKernel, Kernel, CrossStationaryKernel, StationaryKernel, CrossIsotropicKernel,
                      IsotropicKernel, kernel, stationarykernel, isotropickernel, crosskernel,
                      crossstationarykernel, crossisotropickernel)
from ._kernels import Constant, White, ExpQuad, Cauchy, Maternp, Matern, BART
from . import _linalg
from ._GP import GP
from ._fit import empbayes_fit
from ._dist import eval_batch_sharded, eval_concurrent, DistChol
from ._fastraniter import raniter, sample, sample_batch
from . import bayestree
