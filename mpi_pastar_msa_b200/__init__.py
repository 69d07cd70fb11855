"""B200-native data-parallel core of PA-Star (parallel A* multiple sequence alignment).

The product is the C-ABI library ``lib/libpastar_gpu.so`` (hand-written sm_100a CUDA
kernels, include/pastar_gpu.h) and the C++ ``bin/pastar`` CLI.  This Python package is
plumbing for tests, bench.py and the torchrun multi-GPU driver: a ctypes binding that
mirrors the reference's interfaces (Sequences / HeuristicHPair / Node::getNeigh /
Coord::get_id / PAStar::pa_star).  There is no CPU fallback: importing works anywhere,
but every compute call needs the built library and a CUDA device and fails loudly
otherwise.
"""
from .api import (HASH_TYPES, allow_extended_n, release_cached_memory, bench_random_gather, bench_int_peak, PastarError, PastarGPU, default_cost_table, gpu_weights, host_weights, lib_path, load_library, multi_search,  # noqa: F401
                  node_dtype, read_fasta, rescore_alignment, succ_dtype, WEIGHT_DEN, weight_fraction)
