"""plaac_b200 -- B200-native PLAAC per-protein scoring (hot path only).

The product is libplaac_cuda.so (plaac_b200/csrc, C ABI in include/plaac_cuda.h) plus the
C++ host CLI (plaac_b200/host).  This Python package is a thin ctypes binding used by the tests
and bench.py; it has no CPU fallback and raises if the CUDA library is missing.
"""
from .capi import (  # noqa: F401
    LIB_PATH, PlaacError, Params, Summary, SUMMARY_DTYPE, Scorer, default_params, encode, lib, pack,
    RESIDUE_F64, RESIDUE_U8, MultiScorer, shard_plan, PinnedBuffer, host_register, host_unregister,
    pack_words, pack_append, pack_chars, unpack_words, Hits, HITS_CORE, HITS_TOPK, PACK_PER_WORD, Variants, Segments, saturation,
    EFFECT_COLUMNS, effects_dtype, saturation_map, NULL_COLUMNS, Null, shuffle,
    seq_pvalues,
)
