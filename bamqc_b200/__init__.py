"""bamqc_b200 -- B200-native engine for the per-record statistics pass of BamQC's ``bamqualcheck``.

The product is the CUDA/C++ shared library ``libbamqc_b200.so`` (C ABI in ``include/bamqc_b200.h``) and the
``bamqualcheck`` command built from ``bamqc_b200/csrc``.  This package is the thin Python mirror of that
ABI used by the tests, ``bench.py`` and the multi-GPU (torch.distributed / NCCL) merge.
"""
from ._lib import load_library, library_path, build  # noqa: F401
from .engine import Engine, Batch, BamQCError, FIELDS, parse_sam_header  # noqa: F401
from . import synth  # noqa: F401
