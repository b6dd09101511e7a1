"""bore_b200 -- B200-native (sm_100a) implementation of ltiao/bore's BORE-MLP hot path.

Same Python surface as the reference for that path; hand-written CUDA kernels behind a C ABI
(include/bore_b200.h) underneath.  No TensorFlow, no SciPy optimiser, no CPU fallback.
"""
__version__ = "0.1.0"

from .layers import (Dense, Dropout, BinaryCrossentropy, Adam, RMSprop, Adagrad, Adadelta, Adamax, Nadam, L1, L2, L1L2,  # noqa: F401
                     l1, l2, l1_l2)
from .ops import identity, sigmoid, exp, TRANSFORMS  # noqa: F401
from .base import convert, maybe_distort, maybe_distort_batch, truncated_normal  # noqa: F401
from .models import (Sequential, DenseSequential, MaximizableModel,  # noqa: F401
                     MaximizableSequential, MaximizableDenseSequential, BatchMaximizableModel,
                     BatchMaximizableSequential, BatchMaximizableDenseSequential,
                     StackedRecurrentFactory)
from .data import Record, MultiFidelityRecord  # noqa: F401
from .math import steps_per_epoch, ceil_divide  # noqa: F401
from .batched import BatchedMaximizableSequential, problem_shard  # noqa: F401
