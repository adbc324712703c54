"""B200-native create_mega_reads / jf_aligner hot path (see DESIGN.md).

Only what the path needs lives here: csrc/ (CUDA kernels, C ABI, host tools), api.py (ctypes
binding used by tests and bench), tools/ (synthetic input generator).
"""
from .api import (Context, CoordsParams, Index, MrError, Params, Reads, RecordsParams, Result, SrNames, SuperReads, Unitigs,  # noqa: F401
                  default_params, lib, records_params)
