"""microcket_b200 — B200-native (sm_100a) sam2pairs / krmdup / binning hot path of Microcket.

The product is libmicrocket_b200.so (C ABI, include/microcket_b200.h) and the drop-in
executables built next to it.  This package is the thin Python host side used by tests and
bench.py: a ctypes binding that mirrors the C ABI one to one.  There is no CPU fallback:
every compute call raises if the CUDA library or a GPU is missing.
"""
from .capi import (MkError, Lib, lib, build, S2PConfig, Sam2Pairs, Krmdup, PairsWorkspace, synth_host,  # noqa: F401
                   synth_device, synth_opts, SynthOpts, chrom_ranks, Hist, Norm, NormStats, NORM_TYPES, NORM_SCOPES, Xchg, LIB_PATH, PAIR_DTYPE,
                   Bgzf, BgzfMember, bgzf_scan, bgzf_decompress, BgzfDeflate, bgzf_compress, bgzf_deflate_bound, BGZF_EOF)

__all__ = ["MkError", "Lib", "lib", "build", "S2PConfig", "Sam2Pairs", "Krmdup", "PairsWorkspace", "synth_host", "synth_device", "synth_opts", "SynthOpts", "chrom_ranks", "Hist", "Norm", "NormStats", "NORM_TYPES", "NORM_SCOPES", "Xchg", "LIB_PATH", "PAIR_DTYPE", "Bgzf", "BgzfMember", "bgzf_scan", "bgzf_decompress", "BgzfDeflate", "bgzf_compress", "bgzf_deflate_bound", "BGZF_EOF"]
