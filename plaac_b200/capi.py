"""ctypes binding of include/plaac_cuda.h (+ include/plaac_bench.h).

Mirrors the reference's per-protein interface at batch granularity:
  Scorer.score(codes, offsets)          ~ the loop body of scoreallfastas (plaac.java:755-948)
  Scorer.score(..., per_residue=True)   ~ the loop body of plotsomefastas (plaac.java:610-647)
No CPU fallback: if libplaac_cuda.so is not built, importing `lib()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libplaac_cuda.so")

NAA = 22
LUT_LEN = 4001
AANAMES = "XACDEFGHIKLMNPQRSTVWY*"


class PlaacError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libplaac_cuda error {code}: {msg}")
        self.code = code


class Params(C.Structure):
    _fields_ = [
        ("core_len", C.c_int32), ("ww1", C.c_int32), ("ww2", C.c_int32), ("ww3", C.c_int32),
        ("adjust_prolines", C.c_int32), ("mw_window", C.c_int32), ("reserved", C.c_int32 * 2),
        ("lt", (C.c_double * 2) * 2), ("li", C.c_double * 2), ("lf", C.c_double * 2),
        ("le", (C.c_double * NAA) * 2),
        ("le0", C.c_double * NAA), ("llr", C.c_double * NAA), ("papa_lod", C.c_double * NAA),
        ("hydro2", C.c_double * NAA), ("charge", C.c_double * NAA), ("fi_cc", C.c_double * 3),
        ("big_neg", C.c_double), ("ln2", C.c_double), ("loglut", C.c_double * LUT_LEN),
    ]


class Summary(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "mw_score", "mw_start", "mw_end", "llr_start", "llr_end", "vit_maxrun", "core_start", "core_end",
        "prd_start", "prd_end", "prot_len", "fi_numaa", "fi_maxrun", "papa_center")] + [(n, C.c_double) for n in (
        "llr", "core_score", "prd_score", "hmm_all", "hmm_vit", "fi_meanhydro", "fi_meancharge", "fi_meancombo",
        "papa_combo", "papa_prop", "papa_fi", "papa_llr", "papa_llr2")]


assert C.sizeof(Summary) == 160
SUMMARY_DTYPE = np.dtype([(n, "<i4" if t is C.c_int32 else "<f8") for n, t in Summary._fields_])
assert SUMMARY_DTYPE.itemsize == 160

RESIDUE_U8 = ("vit", "map")
RESIDUE_F64 = ("charge", "hydro", "fi", "plaac", "papa", "fix2", "plaacx2", "papax2", "post_bg", "post_prd")


class ResidueOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in RESIDUE_U8 + RESIDUE_F64]


class Stats(C.Structure):
    _fields_ = [("kernel_launches", C.c_int64), ("score_launches", C.c_int64), ("last_total_ms", C.c_float),
                ("last_score_ms", C.c_float), ("last_padded_slots", C.c_int64), ("long_proteins", C.c_int64),
                ("long_redone_chunks", C.c_int64)]


class FastaIndex(C.Structure):
    _fields_ = [("nrec", C.c_int64), ("nres", C.c_int64)]


HITS_CORE, HITS_TOPK = 1, 2
PACK_PER_WORD = 7


class Hits(C.Structure):
    _fields_ = [("mode", C.c_int32), ("rank_flags", C.c_int32), ("capacity", C.c_int64), ("records", C.c_void_p),
                ("index", C.c_void_p), ("count", C.c_int64), ("n_core", C.c_int64)]


class Variants(C.Structure):
    _fields_ = [("nvar", C.c_int64), ("protein", C.c_void_p), ("first_sub", C.c_void_p), ("pos", C.c_void_p),
                ("code", C.c_void_p)]


assert C.sizeof(Variants) == 40


class Segments(C.Structure):
    _fields_ = [("capacity", C.c_int64), ("first", C.c_void_p), ("start", C.c_void_p), ("end", C.c_void_p),
                ("score", C.c_void_p), ("count", C.c_int64)]


assert C.sizeof(Segments) == 48

# Effect columns of plaac_score_variant_effects in bit order (PLAAC_EFFECT_*): the doubles of the record, then the
# CORE change (+1 gained, -1 lost, 0 unchanged).
EFFECT_COLUMNS = tuple(n for n, t in Summary._fields_ if t is C.c_double) + ("core_change",)
assert len(EFFECT_COLUMNS) == 14


class Null(C.Structure):
    _fields_ = [("replicates", C.c_int64), ("seed", C.c_uint64), ("columns", C.c_int32), ("reserved", C.c_int32),
                ("nsel", C.c_int64), ("proteins", C.c_void_p), ("counts", C.c_void_p), ("values", C.c_void_p)]


assert C.sizeof(Null) == 56

# Columns of plaac_score_shuffles in bit order: the doubles of the record (bits 0..12, as EFFECT_COLUMNS), then the
# replicates that have a CORE (PLAAC_NULL_HAS_CORE).
NULL_COLUMNS = EFFECT_COLUMNS[:13] + ("has_core",)

_lib = None


def lib():
    """Load libplaac_cuda.so; raises (no fallback) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PlaacError(-5, f"{LIB_PATH} is missing: run `python -m plaac_b200.build` (there is no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        vp, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_double
        L.plaac_device_count.restype = C.c_int
        L.plaac_create.restype = C.c_int
        L.plaac_create.argtypes = [C.POINTER(vp), C.c_int, C.POINTER(Params)]
        L.plaac_destroy.restype = None
        L.plaac_destroy.argtypes = [vp]
        L.plaac_last_error.restype = C.c_char_p
        L.plaac_last_error.argtypes = [vp]
        L.plaac_score.restype = C.c_int
        L.plaac_score.argtypes = [vp, vp, vp, i64, vp, C.POINTER(ResidueOut)]
        L.plaac_score_device.restype = C.c_int
        L.plaac_score_device.argtypes = [vp, vp, vp, i64, i64, vp, C.POINTER(ResidueOut)]
        L.plaac_sync.restype = C.c_int
        L.plaac_sync.argtypes = [vp]
        L.plaac_stream.restype = vp
        L.plaac_stream.argtypes = [vp]
        L.plaac_params_init.restype = C.c_int
        L.plaac_params_init.argtypes = [C.POINTER(Params), dbl, vp, vp, i32, i32, i32, i32, i32, vp]
        L.plaac_encode_host.restype = None
        L.plaac_encode_host.argtypes = [vp, i64, vp]
        for nm, at in (("plaac_host_alloc", [C.POINTER(vp), C.c_size_t, C.c_int]), ("plaac_host_free", [vp]),
                       ("plaac_host_register", [vp, C.c_size_t]), ("plaac_host_unregister", [vp])):
            getattr(L, nm).restype = C.c_int
            getattr(L, nm).argtypes = at
        L.plaac_set_chunk.restype = C.c_int
        L.plaac_set_chunk.argtypes = [vp, i64, i64]
        L.plaac_set_long_path.restype = C.c_int
        L.plaac_set_long_path.argtypes = [vp, i64, C.c_int]
        L.plaac_set_kernel_variant.restype = C.c_int
        L.plaac_set_kernel_variant.argtypes = [vp, C.c_int]
        L.plaac_get_stats.restype = C.c_int
        L.plaac_get_stats.argtypes = [vp, C.POINTER(Stats)]
        L.plaac_ingest_fasta.restype = C.c_int
        L.plaac_ingest_fasta.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, i64, C.POINTER(FastaIndex), vp]
        L.plaac_ingest_fasta_device.restype = C.c_int
        L.plaac_ingest_fasta_device.argtypes = [vp, vp, i64, vp, vp, vp, vp, vp, i64, C.POINTER(FastaIndex), vp]
        L.plaac_shard_plan.restype = C.c_int
        L.plaac_shard_plan.argtypes = [vp, i64, C.c_int, vp]
        L.plaac_score_multi.restype = C.c_int
        L.plaac_score_multi.argtypes = [C.POINTER(vp), C.c_int, vp, vp, i64, vp, C.POINTER(ResidueOut)]
        L.plaac_score_fasta.restype = C.c_int
        L.plaac_score_fasta.argtypes = [vp, vp, i64, i64, vp, vp, vp, vp, vp, vp, C.POINTER(FastaIndex), vp]
        L.plaac_rank.restype = C.c_int
        L.plaac_rank.argtypes = [vp, vp, i64, C.c_int, vp, C.POINTER(i64)]
        L.plaac_rank_device.restype = C.c_int
        L.plaac_rank_device.argtypes = [vp, vp, i64, C.c_int, vp, C.POINTER(i64)]
        L.plaac_gather_device.restype = C.c_int
        L.plaac_gather_device.argtypes = [vp, vp, vp, i64, vp]
        L.plaac_packed_words.restype = i64
        L.plaac_packed_words.argtypes = [i64]
        L.plaac_pack_host.restype = C.c_int
        L.plaac_pack_host.argtypes = [vp, i64, vp, C.c_int]
        L.plaac_pack_append_host.restype = C.c_int
        L.plaac_pack_append_host.argtypes = [vp, i64, vp, i64, C.c_int]
        L.plaac_pack_chars_host.restype = C.c_int
        L.plaac_pack_chars_host.argtypes = [vp, i64, vp, C.c_int]
        L.plaac_unpack_host.restype = C.c_int
        L.plaac_unpack_host.argtypes = [vp, i64, i64, vp]
        L.plaac_score_packed.restype = C.c_int
        L.plaac_score_packed.argtypes = [vp, vp, vp, i64, i64, vp, C.POINTER(ResidueOut), C.POINTER(Hits)]
        L.plaac_score_multi_packed.restype = C.c_int
        L.plaac_score_multi_packed.argtypes = [C.POINTER(vp), C.c_int, vp, vp, i64, i64, vp, C.POINTER(ResidueOut), C.POINTER(Hits)]
        L.plaac_score_hits.restype = C.c_int
        L.plaac_score_variants.restype = C.c_int
        L.plaac_score_variants.argtypes = [vp, vp, vp, i64, C.POINTER(Variants), vp]
        L.plaac_score_variant_effects.restype = C.c_int
        L.plaac_score_variant_effects.argtypes = [vp, vp, vp, i64, C.POINTER(Variants), i32, vp, vp]
        L.plaac_score_hits.argtypes = [vp, vp, vp, i64, C.POINTER(Hits)]
        L.plaac_score_segments.restype = C.c_int
        L.plaac_score_segments.argtypes = [vp, vp, vp, i64, vp, C.POINTER(Segments)]
        L.plaac_score_shuffles.restype = C.c_int
        L.plaac_score_shuffles.argtypes = [vp, vp, vp, i64, C.POINTER(Null), vp]
        L.plaac_score_shuffles_seq.restype = C.c_int
        L.plaac_score_shuffles_seq.argtypes = [vp, vp, vp, i64, C.POINTER(Null), i64, vp, vp]
        L.plaac_score_shuffles_multi.restype = C.c_int
        L.plaac_score_shuffles_multi.argtypes = [C.POINTER(vp), C.c_int, vp, vp, i64, C.POINTER(Null), vp]
        L.plaac_score_shuffles_seq_multi.restype = C.c_int
        L.plaac_score_shuffles_seq_multi.argtypes = [C.POINTER(vp), C.c_int, vp, vp, i64, C.POINTER(Null), i64, vp, vp]
        L.plaac_shuffle_host.restype = C.c_int
        L.plaac_shuffle_host.argtypes = [vp, i64, C.c_uint64, i64, i64, vp]
        L.plaac_bench_synth_lengths.restype = C.c_int
        L.plaac_bench_synth_lengths.argtypes = [vp, C.c_uint64, i64, i64, dbl, dbl, i32, i32, vp]
        L.plaac_bench_synth_residues.restype = C.c_int
        L.plaac_bench_synth_residues.argtypes = [vp, C.c_uint64, i64, i64, vp, vp, vp, dbl, dbl, vp]
        L.plaac_bench_fp64_peak.restype = C.c_int
        L.plaac_bench_fp64_peak.argtypes = [C.c_int, C.c_int, C.POINTER(dbl), C.POINTER(C.c_float)]
        _lib = L
    return _lib


def default_params(alpha=1.0, bg_counts=None, fg_freq=None, core_len=60, ww1=41, ww2=41, ww3=None,
                   adjust_prolines=True, return_info=False):
    """plaac.java main :310-518 through plaac_params_init (host C++ code, not the oracle)."""
    P = Params()
    if ww3 is None:
        ww3 = ww2  # plaac.java:355
    bgp = fgp = None
    if bg_counts is not None:
        bg = np.ascontiguousarray(bg_counts, dtype=np.float64)
        assert bg.shape == (NAA,)
        bgp = bg.ctypes.data
    if fg_freq is not None:
        fg = np.ascontiguousarray(fg_freq, dtype=np.float64)
        assert fg.shape == (NAA,)
        fgp = fg.ctypes.data
    info = np.zeros((4, NAA))
    rc = lib().plaac_params_init(C.byref(P), float(alpha), bgp, fgp, core_len, ww1, ww2, ww3,
                                 int(bool(adjust_prolines)), info.ctypes.data)
    if rc != 0:
        raise PlaacError(rc, "plaac_params_init failed")
    return (P, info) if return_info else P


def encode(seq, strip_stop=True) -> np.ndarray:
    """string2aa (plaac.java:1764) after the terminal '*' strip of :758, via plaac_encode_host."""
    if isinstance(seq, str):
        seq = seq.encode("latin-1")
    if strip_stop and seq[-1:] == b"*":
        seq = seq[:-1]
    src = np.frombuffer(seq, dtype=np.uint8)
    out = np.empty(len(src), dtype=np.uint8)
    if len(src):
        lib().plaac_encode_host(src.ctypes.data, len(src), out.ctypes.data)
    return out


def pack(seqs):
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    offsets = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    codes = np.concatenate(seqs).astype(np.uint8) if len(seqs) and offsets[-1] > 0 else np.zeros(0, np.uint8)
    return np.ascontiguousarray(codes), offsets


def pack_words(codes: np.ndarray, nthreads: int = 0, out: np.ndarray | None = None) -> np.ndarray:
    """plaac_pack_host: one-byte codes -> radix-22 words (7 residues per uint32) for Scorer.score_packed()."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    nw = int(lib().plaac_packed_words(len(codes)))
    words = out if out is not None else np.zeros(nw, dtype=np.uint32)
    assert words.dtype == np.uint32 and len(words) >= nw
    rc = lib().plaac_pack_host(codes.ctypes.data if len(codes) else None, len(codes), words.ctypes.data if nw else None, nthreads)
    if rc != 0:
        raise PlaacError(rc, "plaac_pack_host: residue code > 21")
    return words


def pack_append(codes: np.ndarray, words: np.ndarray, pos: int, nthreads: int = 0) -> int:
    """plaac_pack_append_host: packs `codes` at residue positions [pos, pos + len) of the batch held in `words`; returns
    the position after them."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    assert words.dtype == np.uint32 and len(words) >= lib().plaac_packed_words(pos + len(codes))
    rc = lib().plaac_pack_append_host(codes.ctypes.data if len(codes) else None, len(codes), words.ctypes.data, pos, nthreads)
    if rc != 0:
        raise PlaacError(rc, "plaac_pack_append_host: residue code > 21")
    return pos + len(codes)


def pack_chars(text: bytes, nthreads: int = 0) -> np.ndarray:
    """plaac_pack_chars_host: FASTA letters -> radix-22 words (aatoint fused with the packing)."""
    buf = np.frombuffer(text, dtype=np.uint8)
    words = np.zeros(int(lib().plaac_packed_words(len(buf))), dtype=np.uint32)
    rc = lib().plaac_pack_chars_host(buf.ctypes.data if len(buf) else None, len(buf), words.ctypes.data if len(words) else None, nthreads)
    if rc != 0:
        raise PlaacError(rc, "plaac_pack_chars_host failed")
    return words


def unpack_words(words: np.ndarray, first: int, count: int) -> np.ndarray:
    words = np.ascontiguousarray(words, dtype=np.uint32)
    out = np.zeros(count, dtype=np.uint8)
    rc = lib().plaac_unpack_host(words.ctypes.data if len(words) else None, first, count, out.ctypes.data if count else None)
    if rc != 0:
        raise PlaacError(rc, "plaac_unpack_host failed")
    return out


class PinnedBuffer:
    """Page-locked host memory from plaac_host_alloc as a numpy array (`.array`); freed by close() / the context
    manager / garbage collection.  Hand `.array` (or slices of it) to Scorer.score()."""

    def __init__(self, shape, dtype=np.uint8, write_combined=False):
        self.dtype = np.dtype(dtype)
        self.shape = (int(shape),) if np.isscalar(shape) else tuple(int(x) for x in shape)
        nbytes = int(np.prod(self.shape, dtype=np.int64)) * self.dtype.itemsize
        p = C.c_void_p()
        rc = lib().plaac_host_alloc(C.byref(p), nbytes, 1 if write_combined else 0)
        if rc != 0:
            raise PlaacError(rc, lib().plaac_last_error(None).decode())
        self.ptr = p.value
        self.nbytes = nbytes
        raw = (C.c_uint8 * max(1, nbytes)).from_address(self.ptr)
        self.array = np.frombuffer(raw, dtype=self.dtype, count=nbytes // self.dtype.itemsize).reshape(self.shape)

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib().plaac_host_free(self.ptr)
            self.ptr = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def host_register(arr: np.ndarray):
    """Pins the memory of an existing contiguous numpy array (plaac_host_register); undo with host_unregister."""
    rc = lib().plaac_host_register(arr.ctypes.data, arr.nbytes)
    if rc != 0:
        raise PlaacError(rc, lib().plaac_last_error(None).decode())


def host_unregister(arr: np.ndarray):
    rc = lib().plaac_host_unregister(arr.ctypes.data)
    if rc != 0:
        raise PlaacError(rc, lib().plaac_last_error(None).decode())


class Scorer:
    """One ctx on one GPU (plaac_create .. plaac_destroy)."""

    def __init__(self, params: Params | None = None, device: int = 0):
        self.params = params if params is not None else default_params()
        self._h = C.c_void_p()
        rc = lib().plaac_create(C.byref(self._h), device, C.byref(self.params))
        if rc != 0:
            raise PlaacError(rc, lib().plaac_last_error(None).decode())
        self.device = device

    def close(self):
        if self._h:
            lib().plaac_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise PlaacError(rc, lib().plaac_last_error(self._h).decode())

    # ---- host buffers (numpy, or pinned torch tensors through .data_ptr()) ----
    def score(self, codes: np.ndarray, offsets: np.ndarray, per_residue: bool = False, summaries: bool = True):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        nprot = len(offsets) - 1
        out = np.zeros(nprot, dtype=SUMMARY_DTYPE) if summaries else None
        res = None
        ro = None
        if per_residue:
            ntot = int(offsets[-1] - offsets[0])
            res = {n: np.zeros(ntot, dtype=np.uint8) for n in RESIDUE_U8}
            res.update({n: np.zeros(ntot, dtype=np.float64) for n in RESIDUE_F64})
            ro = C.byref(ResidueOut(**{n: a.ctypes.data for n, a in res.items()}))
        self._check(lib().plaac_score(self._h, codes.ctypes.data, offsets.ctypes.data, nprot,
                                      out.ctypes.data if out is not None else None, ro))
        if per_residue:
            return out, res
        return out

    def _hits(self, mode, capacity, records=True):
        cap = max(int(capacity), 0)
        rec = np.zeros(cap, dtype=SUMMARY_DTYPE) if records else None
        idx = np.zeros(cap, dtype=np.int32)
        h = Hits(mode=mode, rank_flags=0, capacity=cap, records=rec.ctypes.data if records and cap else None,
                 index=idx.ctypes.data if cap else None, count=0, n_core=0)
        return h, rec, idx

    def score_packed(self, words: np.ndarray, lengths: np.ndarray, nres: int | None = None, summaries: bool = True,
                     per_residue: bool = False, hits: str | None = None, capacity: int | None = None):
        """plaac_score_packed: radix-22 words + int32 lengths in; the table and / or its ranked head out.
        hits: None, "core" (every protein with a CORE, ranked) or "topk" (first `capacity` rows of the ranking).
        Returns summaries (or None) [, residue dict] [, dict(records, index, n_core)] in that order."""
        words = np.ascontiguousarray(words, dtype=np.uint32)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        nprot = len(lengths)
        if nres is None:
            nres = int(lengths.astype(np.int64).sum())
        out = np.zeros(nprot, dtype=SUMMARY_DTYPE) if summaries else None
        res, ro = None, None
        if per_residue:
            res = {n: np.zeros(nres, dtype=np.uint8) for n in RESIDUE_U8}
            res.update({n: np.zeros(nres, dtype=np.float64) for n in RESIDUE_F64})
            ro = C.byref(ResidueOut(**{n: a.ctypes.data for n, a in res.items()}))
        h = rec = idx = None
        if hits is not None:
            h, rec, idx = self._hits(HITS_CORE if hits == "core" else HITS_TOPK, nprot if capacity is None else capacity)
        self._check(lib().plaac_score_packed(self._h, words.ctypes.data if len(words) else None, lengths.ctypes.data if nprot else None,
                                             nprot, nres, out.ctypes.data if out is not None and nprot else None, ro,
                                             C.byref(h) if h is not None else None))
        ret = [out]
        if per_residue:
            ret.append(res)
        if h is not None:
            ret.append({"records": rec[:h.count], "index": idx[:h.count], "n_core": int(h.n_core)})
        return ret[0] if len(ret) == 1 else tuple(ret)

    def score_hits(self, codes: np.ndarray, offsets: np.ndarray, hits: str = "core", capacity: int | None = None):
        """plaac_score_hits: one-byte codes in, ranked compact output only."""
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        nprot = len(offsets) - 1
        h, rec, idx = self._hits(HITS_CORE if hits == "core" else HITS_TOPK, nprot if capacity is None else capacity)
        self._check(lib().plaac_score_hits(self._h, codes.ctypes.data, offsets.ctypes.data, nprot, C.byref(h)))
        return {"records": rec[:h.count], "index": idx[:h.count], "n_core": int(h.n_core)}

    def score_variants(self, codes: np.ndarray, offsets: np.ndarray, protein: np.ndarray, first_sub: np.ndarray,
                       pos: np.ndarray, code: np.ndarray, out: np.ndarray | None = None) -> np.ndarray:
        """plaac_score_variants: variant v is reference protein protein[v] with the residues at
        pos[first_sub[v]:first_sub[v+1]] replaced by code[...]; returns one record per variant, each the record score()
        gives for the mutated protein.  The variant residues are built on the GPU (see saturation()).  out: optional
        record array (e.g. a PinnedBuffer's) of len(protein) rows."""
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        protein = np.ascontiguousarray(protein, dtype=np.int32)
        first_sub = np.ascontiguousarray(first_sub, dtype=np.int64)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        code = np.ascontiguousarray(code, dtype=np.uint8)
        nvar = len(protein)
        if len(first_sub) != nvar + 1:
            raise ValueError(f"first_sub has {len(first_sub)} entries, expected nvar + 1 = {nvar + 1}")
        if out is None:
            out = np.zeros(nvar, dtype=SUMMARY_DTYPE)
        assert out.dtype == SUMMARY_DTYPE and out.flags.c_contiguous and len(out) == nvar
        v = Variants(nvar=nvar, protein=protein.ctypes.data, first_sub=first_sub.ctypes.data, pos=pos.ctypes.data,
                     code=code.ctypes.data)
        self._check(lib().plaac_score_variants(self._h, codes.ctypes.data, offsets.ctypes.data, len(offsets) - 1,
                                               C.byref(v), out.ctypes.data))
        return out

    def variant_effects(self, codes: np.ndarray, offsets: np.ndarray, protein: np.ndarray, first_sub: np.ndarray,
                        pos: np.ndarray, code: np.ndarray, columns=("core_score", "llr"), wild: bool = False,
                        out: np.ndarray | None = None):
        """plaac_score_variant_effects: the variants of score_variants(), but per variant only the selected columns of its
        record minus those of its wild type's (the record score() gives for reference protein protein[v]); 'core_change'
        is +1 if the variant gains a CORE, -1 if it loses it, 0 otherwise.  columns: names of EFFECT_COLUMNS (the double
        fields of SUMMARY_DTYPE and 'core_change').  Returns a structured array with one f8 field per selected column, in
        the order of EFFECT_COLUMNS whatever the order given; with wild=True, (effects, the reference's records).
        out: optional array of that dtype (e.g. a PinnedBuffer's) of len(protein) rows."""
        if isinstance(columns, str):
            columns = (columns,)
        unknown = [c for c in columns if c not in EFFECT_COLUMNS]
        if unknown or not len(columns):
            raise ValueError(f"effect columns must be a non-empty subset of {EFFECT_COLUMNS}, got {list(columns)}")
        mask = 0
        for c in columns:
            mask |= 1 << EFFECT_COLUMNS.index(c)
        dtype = effects_dtype(mask)
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        protein = np.ascontiguousarray(protein, dtype=np.int32)
        first_sub = np.ascontiguousarray(first_sub, dtype=np.int64)
        pos = np.ascontiguousarray(pos, dtype=np.int32)
        code = np.ascontiguousarray(code, dtype=np.uint8)
        nvar = len(protein)
        if len(first_sub) != nvar + 1:
            raise ValueError(f"first_sub has {len(first_sub)} entries, expected nvar + 1 = {nvar + 1}")
        if out is None:
            out = np.zeros(nvar, dtype=dtype)
        assert out.dtype == dtype and out.flags.c_contiguous and len(out) == nvar
        wt = np.zeros(len(offsets) - 1, dtype=SUMMARY_DTYPE) if wild else None
        v = Variants(nvar=nvar, protein=protein.ctypes.data, first_sub=first_sub.ctypes.data, pos=pos.ctypes.data,
                     code=code.ctypes.data)
        self._check(lib().plaac_score_variant_effects(self._h, codes.ctypes.data, offsets.ctypes.data, len(offsets) - 1,
                                                      C.byref(v), mask, out.ctypes.data,
                                                      wt.ctypes.data if wild else None))
        return (out, wt) if wild else out

    def score_segments(self, codes: np.ndarray, offsets: np.ndarray, summaries: bool = True, capacity: int | None = None):
        """plaac_score_segments: summary mode plus every prion-like segment of each protein's Viterbi parse (maximal runs
        of PrD-state residues).  Returns (records or None, {"first", "start", "end", "score"}): the segments of protein i
        are [first[i], first[i+1]), 0-based with end inclusive, score the PRDscore sum over the segment.  capacity: entries
        to make room for (default nprot); if the batch has more segments, the batch is scored a second time with room
        for all of them."""
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        nprot = len(offsets) - 1
        cap = nprot if capacity is None else int(capacity)
        while True:
            out = np.zeros(nprot, dtype=SUMMARY_DTYPE) if summaries else None
            first = np.zeros(nprot + 1, dtype=np.int64)
            start = np.zeros(max(cap, 0), dtype=np.int32)
            end = np.zeros(max(cap, 0), dtype=np.int32)
            score = np.zeros(max(cap, 0), dtype=np.float64)
            sg = Segments(capacity=cap, first=first.ctypes.data, start=start.ctypes.data if cap > 0 else None,
                          end=end.ctypes.data if cap > 0 else None, score=score.ctypes.data if cap > 0 else None, count=0)
            self._check(lib().plaac_score_segments(self._h, codes.ctypes.data, offsets.ctypes.data if nprot >= 0 else None,
                                                   nprot, out.ctypes.data if out is not None and nprot else None,
                                                   C.byref(sg)))
            if sg.count <= cap:
                break
            cap = int(sg.count)
        n = int(sg.count)
        return out, {"first": first, "start": start[:n], "end": end[:n], "score": score[:n]}

    def shuffle_null(self, codes: np.ndarray, offsets: np.ndarray, replicates: int, seed: int = 0,
                     columns=("core_score", "llr", "hmm_all"), proteins=None, values: bool = False, observed: bool = False):
        """plaac_score_shuffles: scores `replicates` (K) composition-preserving shuffles of each selected protein (all of
        them, or the reference indices in `proteins`, which may repeat), built on the GPU, and counts per protein the
        replicates that reach its observed score.  A replicate counts for a double column when its value, NaN taken as
        -Inf, is >= the observed one; 'has_core' counts the replicates with a CORE.  The empirical p-value of a column is
        (1 + count) / (1 + K).  columns: names of NULL_COLUMNS.  Returns a structured array of one int64 field per
        selected column, in the order of NULL_COLUMNS whatever the order given, one row per selected protein; with
        values=True also the replicates' values as an (nsel, K) structured array of f8 fields (has_core: 0 or 1); with
        observed=True also the selected proteins' records (those of score()).  Replicate r of protein i is
        shuffle(codes, offsets, i, r, seed)."""
        a = _NullArgs(codes, offsets, replicates, seed, columns, proteins, observed, values=values)
        self._check(lib().plaac_score_shuffles(self._h, *a.head(), a.obs_ptr))
        return a.fixed_result()

    def shuffle_null_seq(self, codes: np.ndarray, offsets: np.ndarray, max_replicates: int, stop_hits: int = 10, seed: int = 0,
                         columns=("core_score", "llr", "hmm_all"), proteins=None, observed: bool = False):
        """plaac_score_shuffles_seq: the sequential null of Besag and Clifford.  The replicates of shuffle_null are scored
        in order, and a protein's column stops once `stop_hits` (h) of them have reached the observed score, after at
        most `max_replicates` (K_max).  Returns (counts, scored): structured int64 arrays with one field per selected
        column in NULL_COLUMNS order, one row per selected protein; counts is h for a column that stopped and below h
        otherwise, scored is the number of replicates that count covers (K_max if the column did not stop).  With
        observed=True also the selected proteins' records (those of score()).  seq_pvalues turns them into p-values."""
        a = _NullArgs(codes, offsets, max_replicates, seed, columns, proteins, observed, stop_hits=stop_hits)
        self._check(lib().plaac_score_shuffles_seq(self._h, *a.head(), a.h, a.scored.ctypes.data, a.obs_ptr))
        return a.seq_result()

    def score_ptr(self, codes_ptr: int, offsets_ptr: int, nprot: int, summaries_ptr: int):
        """Raw host pointers (e.g. pinned torch tensors)."""
        self._check(lib().plaac_score(self._h, codes_ptr, offsets_ptr, nprot, summaries_ptr, None))

    # ---- device buffers ----
    def score_device(self, d_codes_ptr: int, d_offsets_ptr: int, nprot: int, ntotal: int, d_summaries_ptr: int,
                     residue_ptrs: dict | None = None, sync: bool = True):
        ro = None
        if residue_ptrs is not None:
            ro = C.byref(ResidueOut(**residue_ptrs))
        self._check(lib().plaac_score_device(self._h, d_codes_ptr, d_offsets_ptr, nprot, ntotal, d_summaries_ptr, ro))
        if sync:
            self.sync()

    def ingest_fasta(self, text: bytes, max_rec: int | None = None, bg_counts: bool = False):
        """GPU FASTA ingest (plaac_ingest_fasta): raw file bytes -> dict(codes, offsets, names, flags[, bg_counts]).
        Names are cut from the text with the jar's trimming rule (flag bit 0)."""
        buf = np.frombuffer(text, dtype=np.uint8)
        n = len(buf)
        if max_rec is None:
            max_rec = int(text.count(b">")) + 1
        codes = np.zeros(max(n, 1), dtype=np.uint8)
        offsets = np.zeros(max_rec + 1, dtype=np.int64)
        npos = np.zeros(max(max_rec, 1), dtype=np.int64)
        nlen = np.zeros(max(max_rec, 1), dtype=np.int32)
        flags = np.zeros(max(max_rec, 1) + 8, dtype=np.uint8)
        idx = FastaIndex()
        bg = np.zeros(NAA, dtype=np.float64) if bg_counts else None
        self._check(lib().plaac_ingest_fasta(self._h, buf.ctypes.data if n else None, n, codes.ctypes.data, offsets.ctypes.data,
                                             npos.ctypes.data, nlen.ctypes.data, flags.ctypes.data, max_rec, C.byref(idx),
                                             bg.ctypes.data if bg is not None else None))
        nrec = int(idx.nrec)
        names = []
        for r in range(nrec):
            nm = text[int(npos[r]):int(npos[r]) + int(nlen[r])]
            if flags[r] & 1:  # String.trim() of the whole '>' line: only the tail can change
                nm = nm.rstrip(b"".join(bytes([c]) for c in range(33)))
            names.append(nm.decode("latin-1"))
        out = {"codes": codes[:int(idx.nres)], "offsets": offsets[:nrec + 1], "names": names, "flags": flags[:nrec]}
        if bg is not None:
            out["bg_counts"] = bg
        return out

    def rank(self, summaries: np.ndarray):
        """plaac_rank: the web front end's order (web/lib/server.rb:222-229) -> (order int32[nprot], n_core)."""
        summaries = np.ascontiguousarray(summaries, dtype=SUMMARY_DTYPE)
        order = np.zeros(len(summaries), dtype=np.int32)
        ncore = C.c_int64(0)
        self._check(lib().plaac_rank(self._h, summaries.ctypes.data, len(summaries), 0,
                                     order.ctypes.data, C.byref(ncore)))
        return order, int(ncore.value)

    def rank_device(self, d_summaries_ptr: int, nprot: int, d_order_ptr: int) -> int:
        ncore = C.c_int64(0)
        self._check(lib().plaac_rank_device(self._h, d_summaries_ptr, nprot, 0,
                                            d_order_ptr, C.byref(ncore)))
        return int(ncore.value)

    def gather_device(self, d_summaries_ptr: int, d_order_ptr: int, count: int, d_out_ptr: int, sync: bool = True):
        self._check(lib().plaac_gather_device(self._h, d_summaries_ptr, d_order_ptr, count, d_out_ptr))
        if sync:
            self._check(lib().plaac_sync(self._h))

    def set_chunk(self, max_residues=0, max_proteins=0):
        self._check(lib().plaac_set_chunk(self._h, max_residues, max_proteins))

    def set_long_path(self, min_len: int, warm: int = 0):
        """plaac_set_long_path: length threshold of the chunked long-sequence path (0 = off, -1 = automatic); warm:
        warm-up residues of its chunks (0 keeps the current value, a negative value is taken by its magnitude; -1 gives
        the shortest warm-up, with which nearly every chunk is redone sequentially)."""
        self._check(lib().plaac_set_long_path(self._h, min_len, warm))

    def set_kernel_variant(self, variant: int):
        """0 auto, 1 reference-order anchor kernel, 2 throughput kernel."""
        self._check(lib().plaac_set_kernel_variant(self._h, variant))

    def sync(self):
        self._check(lib().plaac_sync(self._h))

    def stream(self) -> int:
        return int(lib().plaac_stream(self._h) or 0)

    def stats(self) -> Stats:
        s = Stats()
        self._check(lib().plaac_get_stats(self._h, C.byref(s)))
        return s


SATURATION_CODES = np.arange(1, 21, dtype=np.uint8)  # A C D E F G H I K L M N P Q R S T V W Y


def saturation(codes: np.ndarray, offsets: np.ndarray, proteins=None):
    """Every single substitution of the given reference proteins (default: all), as the four arrays of
    Scorer.score_variants: (protein, first_sub, pos, code).  Per protein: the wild type first, then the positions in
    ascending order, at each one every code 1..20 (A C D E F G H I K L M N P Q R S T V W Y) other than the residue
    there (all 20 if that residue is X or '*')."""
    codes = np.asarray(codes, dtype=np.uint8)
    offsets = np.asarray(offsets, dtype=np.int64)
    if proteins is None:
        proteins = np.arange(len(offsets) - 1)
    proteins = np.asarray(proteins, dtype=np.int64)
    parts_prot, parts_pos, parts_code = [], [], []
    for p in proteins:
        ref = codes[offsets[p]:offsets[p + 1]]
        alt = np.broadcast_to(SATURATION_CODES, (len(ref), 20))
        keep = alt != ref[:, None]  # (a residue outside 1..20 keeps all 20)
        pos = np.broadcast_to(np.arange(len(ref), dtype=np.int32)[:, None], (len(ref), 20))[keep]
        parts_pos.append(pos)
        parts_code.append(alt[keep])
        parts_prot.append(np.full(len(pos) + 1, p, dtype=np.int32))
    if not parts_prot:
        return np.zeros(0, np.int32), np.zeros(1, np.int64), np.zeros(0, np.int32), np.zeros(0, np.uint8)
    protein = np.concatenate(parts_prot)
    pos = np.concatenate(parts_pos)
    code = np.concatenate(parts_code)
    # the wild type of each protein has no substitution, every other variant one
    nsub = np.concatenate([np.r_[0, np.ones(len(x), np.int64)] for x in parts_pos])
    first_sub = np.zeros(len(protein) + 1, dtype=np.int64)
    np.cumsum(nsub, out=first_sub[1:])
    return protein, first_sub, np.ascontiguousarray(pos, dtype=np.int32), np.ascontiguousarray(code, dtype=np.uint8)


def shuffle(codes: np.ndarray, offsets: np.ndarray, protein: int, replicate: int, seed: int = 0) -> np.ndarray:
    """plaac_shuffle_host: replicate `replicate` of protein `protein` of the batch (codes, offsets), exactly as
    Scorer.shuffle_null builds it on the GPU: a permutation of the protein's residues.  No GPU needed."""
    codes = np.ascontiguousarray(codes, dtype=np.uint8)
    a, b = int(offsets[protein]), int(offsets[protein + 1])
    src = np.ascontiguousarray(codes[a:b])
    out = np.empty(b - a, dtype=np.uint8)
    rc = lib().plaac_shuffle_host(src.ctypes.data, b - a, int(seed) & (2**64 - 1), int(protein), int(replicate),
                                  out.ctypes.data)
    if rc != 0:
        raise PlaacError(rc, lib().plaac_last_error(None).decode())
    return out


def _null_mask(columns):
    """Column names of the shuffle nulls -> (PLAAC_EFFECT_* / PLAAC_NULL_HAS_CORE mask, the names in bit order)."""
    if isinstance(columns, str):
        columns = (columns,)
    unknown = [c for c in columns if c not in NULL_COLUMNS]
    if unknown or not len(columns):
        raise ValueError(f"null columns must be a non-empty subset of {NULL_COLUMNS}, got {list(columns)}")
    mask = 0
    for c in columns:
        mask |= 1 << NULL_COLUMNS.index(c)
    return mask, [n for k, n in enumerate(NULL_COLUMNS) if mask >> k & 1]


class _NullArgs:
    """The argument handling Scorer's and MultiScorer's shuffle nulls share: the checks (ValueError before any call),
    the Null spec and the output arrays."""

    def __init__(self, codes, offsets, replicates, seed, columns, proteins, observed, values=False, stop_hits=None):
        mask, names = _null_mask(columns)
        K = int(replicates)
        if stop_hits is not None:
            self.h = int(stop_hits)
            if self.h < 1:
                raise ValueError(f"stop_hits must be >= 1, got {self.h}")
            if K < 0:
                raise ValueError(f"max_replicates must be >= 0, got {K}")
        self.codes = np.ascontiguousarray(codes, dtype=np.uint8)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.nprot = len(self.offsets) - 1
        self.sel = None if proteins is None else np.ascontiguousarray(proteins, dtype=np.int32)
        nsel = self.nprot if self.sel is None else len(self.sel)
        self.counts = np.zeros(nsel, dtype=[(n, "<i8") for n in names])
        self.scored = np.zeros(nsel, dtype=self.counts.dtype) if stop_hits is not None else None
        self.vals = np.zeros((nsel, max(K, 0)), dtype=[(n, "<f8") for n in names]) if values else None
        self.obs = np.zeros(nsel, dtype=SUMMARY_DTYPE) if observed else None
        self.obs_ptr = self.obs.ctypes.data if observed else None
        self.null = Null(replicates=K, seed=int(seed) & (2**64 - 1), columns=mask, reserved=0,
                         nsel=-1 if self.sel is None else nsel, proteins=self.sel.ctypes.data if self.sel is not None else None,
                         counts=self.counts.ctypes.data, values=self.vals.ctypes.data if values else None)

    def head(self):
        """The arguments after the ctx(s): codes, offsets, nprot, null_spec."""
        return self.codes.ctypes.data, self.offsets.ctypes.data, self.nprot, C.byref(self.null)

    def fixed_result(self):
        ret = [self.counts] + ([self.vals] if self.vals is not None else []) + ([self.obs] if self.obs is not None else [])
        return ret[0] if len(ret) == 1 else tuple(ret)

    def seq_result(self):
        return (self.counts, self.scored, self.obs) if self.obs is not None else (self.counts, self.scored)


def seq_pvalues(counts: np.ndarray, scored: np.ndarray, stop_hits: int, max_replicates: int) -> np.ndarray:
    """The p-values of Scorer.shuffle_null_seq's (counts, scored): h / L where a column stopped (count == h), else
    (count + 1) / (K_max + 1).  One float64 field per double column; has_core is left out, as the CLI leaves out its p."""
    h, K = int(stop_hits), int(max_replicates)
    names = [n for n in counts.dtype.names if n != "has_core"]
    out = np.zeros(len(counts), dtype=[(n, "<f8") for n in names])
    for n in names:
        c, L = counts[n].astype(np.float64), scored[n].astype(np.float64)
        stopped = counts[n] == h
        out[n] = np.where(stopped, h / np.where(stopped, L, 1.0), (c + 1.0) / (K + 1.0))
    return out


def effects_dtype(columns: int) -> np.dtype:
    """The row of plaac_score_variant_effects for a PLAAC_EFFECT_* mask: one f8 field per set bit, in bit order."""
    return np.dtype([(n, "<f8") for k, n in enumerate(EFFECT_COLUMNS) if columns >> k & 1])


def saturation_map(effects_column: np.ndarray, codes: np.ndarray, offsets: np.ndarray, proteins=None):
    """One effect column of a scan built by saturation(codes, offsets, proteins) (e.g. variant_effects(...)['llr']) as
    the scan's heat maps: per protein an (n, 20) array, row i = position i, columns A C D E F G H I K L M N P Q R S T V W
    Y (SATURATION_CODES), with NaN in the cell of the residue already there.  The wild-type row of each protein is left
    out."""
    codes = np.asarray(codes, dtype=np.uint8)
    offsets = np.asarray(offsets, dtype=np.int64)
    if proteins is None:
        proteins = np.arange(len(offsets) - 1)
    col = np.asarray(effects_column, dtype=np.float64)
    maps, at = [], 0
    for p in np.asarray(proteins, dtype=np.int64):
        ref = codes[offsets[p]:offsets[p + 1]]
        keep = SATURATION_CODES[None, :] != ref[:, None]
        nsub = int(keep.sum())
        if at + 1 + nsub > len(col):
            raise ValueError(f"{len(col)} effects are fewer than the scan of these proteins has variants")
        m = np.full((len(ref), 20), np.nan)
        m[keep] = col[at + 1:at + 1 + nsub]  # (row-major: positions ascending, codes ascending, as saturation() lists them)
        maps.append(m)
        at += 1 + nsub
    if at != len(col):
        raise ValueError(f"{len(col)} effects, but the scan of these proteins has {at} variants")
    return maps


def shard_plan(offsets: np.ndarray, nshards: int) -> np.ndarray:
    """plaac_shard_plan: contiguous, residue-balanced shard bounds (nshards+1 protein indices).  Host arithmetic only."""
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    bounds = np.zeros(nshards + 1, dtype=np.int64)
    rc = lib().plaac_shard_plan(offsets.ctypes.data, len(offsets) - 1, nshards, bounds.ctypes.data)
    if rc != 0:
        raise PlaacError(rc, "plaac_shard_plan failed")
    return bounds


class MultiScorer:
    """One ctx per GPU of this box, driven from one process through plaac_score_multi and the multi-GPU shuffle nulls
    (one host thread per GPU)."""

    def __init__(self, params: Params | None = None, devices=None):
        n = lib().plaac_device_count()
        if devices is None:
            devices = list(range(n))
        if not devices:
            raise PlaacError(-5, "no CUDA device (there is no CPU fallback)")
        self.scorers = [Scorer(params, d) for d in devices]

    def close(self):
        for s in self.scorers:
            s.close()
        self.scorers = []

    def _handles(self):
        return (C.c_void_p * len(self.scorers))(*[s._h for s in self.scorers]), len(self.scorers)

    def _check(self, rc):
        """An error's text from every scorer (the call puts it on the ctx it happened on), else the global one."""
        if rc != 0:
            msgs = [lib().plaac_last_error(s._h).decode() for s in self.scorers]
            raise PlaacError(rc, "; ".join(m for m in msgs if m) or lib().plaac_last_error(None).decode())

    def score(self, codes: np.ndarray, offsets: np.ndarray, per_residue: bool = False):
        codes = np.ascontiguousarray(codes, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        nprot = len(offsets) - 1
        out = np.zeros(nprot, dtype=SUMMARY_DTYPE)
        res, ro = None, None
        if per_residue:
            ntot = int(offsets[-1] - offsets[0])
            res = {n: np.zeros(ntot, dtype=np.uint8) for n in RESIDUE_U8}
            res.update({n: np.zeros(ntot, dtype=np.float64) for n in RESIDUE_F64})
            ro = C.byref(ResidueOut(**{n: a.ctypes.data for n, a in res.items()}))
        self._check(lib().plaac_score_multi(*self._handles(), codes.ctypes.data, offsets.ctypes.data, nprot,
                                            out.ctypes.data, ro))
        return (out, res) if per_residue else out

    def score_packed(self, words: np.ndarray, lengths: np.ndarray, per_residue: bool = False, hits: str | None = None,
                     capacity: int | None = None):
        """plaac_score_multi_packed: (summaries[, residue dict][, hits dict])."""
        words = np.ascontiguousarray(words, dtype=np.uint32)
        lengths = np.ascontiguousarray(lengths, dtype=np.int32)
        nprot = len(lengths)
        nres = int(lengths.astype(np.int64).sum())
        out = np.zeros(nprot, dtype=SUMMARY_DTYPE)
        res, ro = None, None
        if per_residue:
            res = {n: np.zeros(nres, dtype=np.uint8) for n in RESIDUE_U8}
            res.update({n: np.zeros(nres, dtype=np.float64) for n in RESIDUE_F64})
            ro = C.byref(ResidueOut(**{n: a.ctypes.data for n, a in res.items()}))
        h = rec = idx = None
        if hits is not None:
            h, rec, idx = self.scorers[0]._hits(HITS_CORE if hits == "core" else HITS_TOPK, nprot if capacity is None else capacity)
        self._check(lib().plaac_score_multi_packed(*self._handles(), words.ctypes.data, lengths.ctypes.data, nprot, nres,
                                                   out.ctypes.data, ro, C.byref(h) if h is not None else None))
        ret = [out]
        if per_residue:
            ret.append(res)
        if h is not None:
            ret.append({"records": rec[:h.count], "index": idx[:h.count], "n_core": int(h.n_core)})
        return ret[0] if len(ret) == 1 else tuple(ret)

    def shuffle_null(self, codes: np.ndarray, offsets: np.ndarray, replicates: int, seed: int = 0,
                     columns=("core_score", "llr", "hmm_all"), proteins=None, values: bool = False, observed: bool = False):
        """plaac_score_shuffles_multi: Scorer.shuffle_null on every GPU, each scoring a range of every protein's
        replicates.  Same arguments, same results, byte for byte."""
        a = _NullArgs(codes, offsets, replicates, seed, columns, proteins, observed, values=values)
        self._check(lib().plaac_score_shuffles_multi(*self._handles(), *a.head(), a.obs_ptr))
        return a.fixed_result()

    def shuffle_null_seq(self, codes: np.ndarray, offsets: np.ndarray, max_replicates: int, stop_hits: int = 10, seed: int = 0,
                         columns=("core_score", "llr", "hmm_all"), proteins=None, observed: bool = False):
        """plaac_score_shuffles_seq_multi: Scorer.shuffle_null_seq with every round's replicates split over the GPUs.
        Same arguments, same results, byte for byte."""
        a = _NullArgs(codes, offsets, max_replicates, seed, columns, proteins, observed, stop_hits=stop_hits)
        self._check(lib().plaac_score_shuffles_seq_multi(*self._handles(), *a.head(), a.h, a.scored.ctypes.data, a.obs_ptr))
        return a.seq_result()
