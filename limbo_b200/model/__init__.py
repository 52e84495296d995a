from .gp import GP, GPBasic, GPOpt  # noqa: F401
from .hp_opt import KernelLFOpt, KernelLooOpt, KernelMeanLFOpt, MeanLFOpt, NoLFOpt, ParallelLFOpt  # noqa: F401
from .multi_gp import MultiGP  # noqa: F401
from .sparsified_gp import SparsifiedGP, sparsify  # noqa: F401
