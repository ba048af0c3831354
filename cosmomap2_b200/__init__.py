"""
cosmomap2_b200 -- B200-native drop-in for the map-making solve of giuspugl/COSMOMAP2.

``from cosmomap2_b200 import *`` gives what the reference's ``from interfaces import *`` +
``from utilities import *`` give for the hot path: the operator classes, ``ProcessTimeSamples``,
the deflation helpers, the BLAS shims and the aliases ``lp`` (operator algebra), ``blk`` and
``spla`` (scipy.sparse.linalg), plus the device-resident ``cg``.

The CUDA library (cosmomap2_b200/csrc/libcosmomap2_b200.so) is loaded at import and there is no
CPU fallback: importing without it raises ImportError, computing without a GPU raises RuntimeError.
"""
import scipy.sparse.linalg as spla  # noqa: F401

from . import _cabi  # noqa: F401  (fails loudly if the shared library is missing)
from . import linop as lp  # noqa: F401
from . import linearoperators as blk  # noqa: F401  (BlockDiagonalLinearOperator lives there)
from .linearoperators import (SparseLO, ToeplitzLO, WeightingLO, BlockLO, FilterLO,  # noqa: F401
                              BlockDiagonalLinearOperator, BlockDiagonalLO,
                              BlockDiagonalPreconditionerLO, InverseLO, CoarseLO, DeflationLO,
                              GroundFilterLO,
                              TwoLevelPreconditionerLO)
from .process_ces import ProcessTimeSamples, BlockWeights  # noqa: F401
from .deflationlib import (arnoldi, build_hess, build_Z, run_krypy_arnoldi,  # noqa: F401
                           find_ritz_eigenvalues, krypy_arnoldi, krypy_ritz, eigsh, scan_coarse_space,
                           coarse_products)
from .utilities import (dgemm, norm2, scalprod, get_legendre_polynomials, is_sorted,  # noqa: F401
                        bash_colors, filter_warnings, angles_gen, pairs_gen, checking_output,
                        noise_val, subscan_resize, system_setup, reorganize_map, profile_run,
                        output_profile, subtract_offset, rescalepixels)
from .pcg import cg  # noqa: F401
from .noise import noise_psd, inverse_noise_bands  # noqa: F401
from . import IOfiles  # noqa: F401
from .IOfiles import (read_from_data, read_multiple_ces, read_from_data_with_subscan_resize,  # noqa: F401
                      read_ces_shard, flagging_subscan, flagging_not_in_allCES,
                      write_ritz_eigenvectors_to_hdf5, read_ritz_eigenvectors_from_hdf5,
                      read_obspix_from_hdf5, write_obspix_to_hdf5, write_to_hdf5, read_from_hdf5,
                      save_maplist, read_maplist, full2cutskymap, obspix2mask, find_common_obspix,
                      write_ces_to_hdf5)

__version__ = "0.1.0"
