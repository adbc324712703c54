"""B200-native create_mega_reads / jf_aligner hot path (see DESIGN.md).

Only what the path needs lives here: csrc/ (CUDA kernels, C ABI, host tools), api.py (ctypes
binding used by tests and bench), tools/ (synthetic input generator).
"""
from .api import (Context, Index, MrError, Params, Reads, RecordsParams, Result, SuperReads, Unitigs, default_params, lib,  # noqa: F401
                  records_params)
