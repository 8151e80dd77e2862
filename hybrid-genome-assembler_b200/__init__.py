"""hga_b200 — B200-native `categorization` hot path (scan -> membership -> incidence -> pair count -> threshold ->
components) behind a C-ABI (include/hga_b200.h). This package is the Python host side: a ctypes binding of
libhga_b200.so (capi) and a mirror of the reference's ReadClusteringEngine stage interface (engine).

There is no CPU path: importing works anywhere (so that the library's exports can be checked), but every compute
entry point raises HgaError unless a CUDA device is present.
"""
from .capi import HgaError, Handle, library_path, load_library, pack_bases  # noqa: F401
from .engine import ReadClusteringConfig, ReadClusteringEngine, load_text_file_kmers, SequenceRecords  # noqa: F401
from . import capi, parallel  # noqa: F401,E402
