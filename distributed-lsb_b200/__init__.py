"""B200-native distributed LSD radix sort: the mySort / globalShuffle hot path of
ronawho/distributed-lsb (mpi/mpi_lsbsort.cpp:481-585) as hand-written sm_100a CUDA kernels
behind the C ABI of include/lsbsort.h.

The directory name carries a hyphen (it mirrors the reference's repository name); import it
through the alias module at the repository root:

    import distributed_lsb_b200 as lsb
"""
from . import hostlogic  # noqa: F401
from .lsbsort import (  # noqa: F401
    ELT,
    DistributedSorter,
    LsbError,
    argsort,
    Stats,
    Verify,
    abi_symbols,
    comm_unique_id,
    header_symbols,
    lexsort,
    library_path,
    load_library,
    sort,
    sort_pairs,
    sort_segments,
    sort_tensor,
    tune,
)
