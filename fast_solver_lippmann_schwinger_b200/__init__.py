"""B200-native hot path of the fast Lippmann-Schwinger solver (libls_cuda.so + host mirror).

Only what the path needs lives here: ``csrc/`` (CUDA kernels + the C ABI of include/ls_cuda.h),
``_lib`` (ctypes binding), ``operators`` / ``krylov`` (the reference's operator interface) and
``sparsifier`` (the preconditioner's stencil matrices sampled through operator applies).
"""
from ._lib import (DeviceBuffer, LSCudaError, LSUnsupported, PinnedArray, declared_symbols, lib)  # noqa: F401
from .operators import FastM, FastM3D, FFTconvolution, apply_batch, batch_cols, fastconvolution, mul_  # noqa: F401
from .krylov import (ConvergenceHistory, GPUMspFactorization, GPUSparseMatrixCSC, KrylovWorkspace,  # noqa: F401
                     SparsifyingPreconditioner, cscmv_, gmres_)
from . import sparsifier  # noqa: F401,E402
