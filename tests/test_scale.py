"""Scoring past the 32-bit size boundaries, against the CPU oracle.

The other GPU tests score at most a few hundred thousand proteins, so every residue offset, record byte offset, chunk
index and ranking position they reach fits in 31 bits.  The tests here score batches where those quantities cross 2^31,
2^32 and 2^24, and compare the results with the oracle (tests/parity.py rules) on the rows around each boundary:

  * the benchmark's own shard (bench.synth_shard: 12.5 M proteins, 4.39 G residues), through every entry point that
    scores it, with the sample `bench.py --dump-outputs` publishes;
  * a batch of 17 M short proteins: more than 2^24 rows to rank and more than 2^31 bytes of records;
  * a FASTA image larger than 2 GiB through the ingest and plaac_score_fasta;
  * a saturation scan of one 34 000-residue protein: 2.2e10 variant residues in one plaac_score_variants call.

Per-residue mode is not run at these sizes (82 bytes out per residue).  The whole shard against the oracle is
scripts/gpu/full_shard_soak.py.  Each test asserts the size it exists for.  The large arrays live in class-scoped
fixtures, so each is freed when its class is done and no two of them are alive at once."""
import ctypes as C
import gc
import math

import numpy as np
import pytest

import bench
import plaac_b200
from oracle import orc
from tests import synth
from tests.test_gpu_parity import _check
from tests.test_ingest import expected as fasta_expected, reference_reader
from tests.test_rank import web_order
from tests.test_variant_effects import assert_same_effects, expected as effects_expected
from tests.test_variants import assert_same_bytes, materialise

NT = bench.host_threads()
BOUNDARY_SPAN = 2_000        # proteins on each side of a boundary protein, and at the end of a batch
RANDOM_SAMPLE = 200_000
ROW_BYTES = plaac_b200.SUMMARY_DTYPE.itemsize


# ---------------------------------------------------------------------------------------------- helpers
def proteins_around(offsets, residue, k):
    """Indices of the protein that holds residue `residue` of the batch and of the k proteins on each side of it (in
    batch order, clipped to the batch).  Empty proteins hold no residue: the protein found is the non-empty one
    that does, and empty proteins beside it count among the k."""
    offsets = np.asarray(offsets, dtype=np.int64)
    nprot = len(offsets) - 1
    assert 0 <= residue < offsets[-1], (residue, int(offsets[-1]))
    i = int(np.searchsorted(offsets, residue, side="right")) - 1
    return np.arange(max(0, i - k), min(nprot, i + k + 1), dtype=np.int64)


def subset(codes, offsets, idx):
    """The proteins idx of a batch as a batch of their own."""
    idx = np.asarray(idx, dtype=np.int64)
    seqs = [codes[offsets[i]:offsets[i + 1]] for i in idx]
    return orc.pack(seqs) if len(seqs) else (np.zeros(0, np.uint8), np.zeros(1, np.int64))


def check_oracle(P, codes, offsets, got_all, idx, what):
    """Records got_all[idx] against the oracle's for the same proteins: tests/parity.py rules, at most one PAPA
    tie-class row per 20 000 rows (and one more)."""
    idx = np.unique(np.asarray(idx, dtype=np.int64))
    c, o = subset(codes, offsets, idx)
    ref = orc.score_batch(P, c, o, nthreads=NT)
    got = np.ascontiguousarray(got_all[idx])
    differs = np.zeros(len(idx), bool)
    for f in orc.INT_FIELDS:
        differs |= got[f] != ref[f]
    where = ", ".join(f"row {i} = protein {idx[i]} at residue {int(offsets[idx[i]])}" for i in np.nonzero(differs)[0][:10])
    _check(got, ref, f"{what} ({len(idx)} proteins; {where})", P, c, o, max_ties=1 + len(idx) // 20_000)
    return len(idx)


def rows(a):
    return np.ascontiguousarray(a).view(np.uint8).reshape(len(a), ROW_BYTES)


def assert_same_records(got, want, what, piece=1 << 20):
    """Byte identity of two record arrays, compared a million rows at a time (no full-size temporaries)."""
    assert len(got) == len(want), (what, len(got), len(want))
    g, w = rows(got), rows(want)
    for lo in range(0, len(g), piece):
        hi = min(len(g), lo + piece)
        bad = np.nonzero((g[lo:hi] != w[lo:hi]).any(axis=1))[0]
        assert len(bad) == 0, f"{what}: {len(bad)} records differ in rows [{lo}, {hi}), first {(lo + bad[:10]).tolist()}"


def device_records(t, nprot):
    return t.cpu().numpy().reshape(-1).view(plaac_b200.SUMMARY_DTYPE)[:nprot]


def release(d):
    import torch

    d.clear()
    gc.collect()
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------- CPU
def test_proteins_around_a_residue():
    # lengths 3, 0, 0, 4, 1, 0, 2: residues 0-2 | - | - | 3-6 | 7 | - | 8-9
    offsets = np.array([0, 3, 3, 3, 7, 8, 8, 10], np.int64)
    assert proteins_around(offsets, 0, 0).tolist() == [0]                      # first residue of the batch
    assert proteins_around(offsets, 2, 0).tolist() == [0]                      # last residue of a protein
    assert proteins_around(offsets, 3, 0).tolist() == [3]                      # first residue, after two empty ones
    assert proteins_around(offsets, 6, 0).tolist() == [3]
    assert proteins_around(offsets, 3, 1).tolist() == [2, 3, 4]                # empty neighbours count
    assert proteins_around(offsets, 3, 2).tolist() == [1, 2, 3, 4, 5]
    assert proteins_around(offsets, 7, 1).tolist() == [3, 4, 5]                # a one-residue protein
    assert proteins_around(offsets, 8, 1).tolist() == [5, 6]                   # an empty one before, clipped after
    assert proteins_around(offsets, 9, 5).tolist() == [1, 2, 3, 4, 5, 6]       # last residue of the batch
    assert proteins_around(offsets, 1, 9).tolist() == list(range(7))
    for bad in (-1, 10):
        with pytest.raises(AssertionError):
            proteins_around(offsets, bad, 1)
    # the same answer as a scan over every residue, on random lengths with many empty proteins
    rng = np.random.default_rng(3)
    lens = rng.integers(0, 4, size=400) * (rng.random(400) < 0.6)
    offsets = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    owner = np.repeat(np.arange(400), lens)
    for r in range(int(offsets[-1])):
        i = int(owner[r])
        assert offsets[i] <= r < offsets[i + 1]
        assert proteins_around(offsets, r, 3).tolist() == list(range(max(0, i - 3), min(400, i + 4)))
    # residues at the boundaries this module samples, in a batch whose offsets cross them
    offsets = np.array([0, 2**31 - 1, 2**31, 2**31, 2**32 - 1, 2**32 + 1, 2**33], np.int64)
    assert proteins_around(offsets, 2**31 - 1, 0).tolist() == [1]
    assert proteins_around(offsets, 2**31, 0).tolist() == [3]
    assert proteins_around(offsets, 2**31, 1).tolist() == [2, 3, 4]
    assert proteins_around(offsets, 2**32 - 1, 0).tolist() == [4]
    assert proteins_around(offsets, 2**32, 0).tolist() == [4]


# ---------------------------------------------------------------------------------------------- 1. the bench shard
@pytest.mark.gpu
class TestBenchShard:
    """Rank 0's shard of bench.py (12.5 M proteins, 4.39 G residues), scored as its timed step scores it."""

    NPROT = 12_500_000

    @pytest.fixture(scope="class")
    def shard(self):
        import torch

        dev = torch.device("cuda", 0)
        codes, offsets, ntotal = bench.synth_shard(plaac_b200.lib(), dev, 0, self.NPROT)
        recs = torch.empty(self.NPROT * ROW_BYTES, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        sc = plaac_b200.Scorer(device=0)
        n0 = sc.stats().long_proteins
        sc.score_device(codes.data_ptr(), offsets.data_ptr(), self.NPROT, ntotal, recs.data_ptr(), sync=True)
        default_long = sc.stats().long_proteins - n0
        sc.close()
        d = dict(d_codes=codes, d_offsets=offsets, d_rec=recs, ntotal=ntotal, default_long=default_long,
                 h_codes=codes[:ntotal].cpu().numpy(), h_offs=offsets.cpu().numpy(), h_rec=device_records(recs, self.NPROT),
                 P=orc.make_params())
        d["lens"] = np.diff(d["h_offs"])
        del codes, offsets, recs
        yield d
        release(d)

    @staticmethod
    def ranking(shard):
        if "order" not in shard:
            shard["order"] = web_order(shard["h_rec"])
        return shard["order"]

    def test_boundaries_long_path_and_published_sample_against_oracle(self, shard, tmp_path):
        import torch

        nprot, ntotal, offs, lens = self.NPROT, shard["ntotal"], shard["h_offs"], shard["lens"]
        assert ntotal > 2**32 and offs[-1] == ntotal
        pick = [proteins_around(offs, r, BOUNDARY_SPAN) for r in (2**31 - 1, 2**31, 2**32 - 1, 2**32)]
        pick.append(np.arange(nprot - BOUNDARY_SPAN, nprot))
        # the proteins the timed call (default threshold, 8 192 residues) sent to the long path, and the longest
        # proteins of the shard, which the long path takes at lower thresholds (test_long_path_past_2_32, and every
        # chunk of the host call in test_host_entry_points_give_the_device_records)
        assert shard["default_long"] == int((lens >= 8192).sum())
        pick.append(np.nonzero(lens >= 8192)[0])
        pick.append(np.argsort(lens, kind="stable")[-150:])
        # the automatic threshold of one device call over the whole shard: only proteins of at least ntotal/81600 + 220
        # residues (include/plaac_cuda.h), which is beyond the shard's longest: none, and the same bytes
        sc = plaac_b200.Scorer(device=0)
        sc.set_long_path(-1)
        auto = torch.empty_like(shard["d_rec"])
        n0 = sc.stats().long_proteins
        sc.score_device(shard["d_codes"].data_ptr(), shard["d_offsets"].data_ptr(), nprot, ntotal, auto.data_ptr(), sync=True)
        n_auto = sc.stats().long_proteins - n0
        sc.close()
        assert torch.equal(auto, shard["d_rec"]), "automatic long-path threshold: records differ from the timed call's"
        del auto
        torch.cuda.empty_cache()
        assert lens.max() < ntotal // 81600 + 220 and n_auto == 0
        print(f"default threshold: {shard['default_long']} long proteins; longest protein {lens.max()} residues")
        # the sample bench.py --dump-outputs publishes, written from the same device records
        bench.dump_outputs(str(tmp_path), shard["d_rec"], 0, nprot)
        idx = np.load(tmp_path / "protein_index.npy").astype(np.int64)
        assert len(idx) == bench.DUMP_PROTEINS and (np.diff(idx) > 0).all() and idx[-1] < nprot
        want = shard["h_rec"][idx]
        for n in plaac_b200.SUMMARY_DTYPE.names:
            got, w = np.load(tmp_path / (n + ".npy")), want[n].astype(np.float64)
            if plaac_b200.SUMMARY_DTYPE[n].kind == "f":
                cls = np.load(tmp_path / (n + "_nonfinite.npy"))
                assert (cls == np.select([np.isnan(w), w == np.inf, w == -np.inf], [1, 2, 3], 0)).all(), n
                w = np.where(cls == 0, w, 0.0)
            assert (got == w).all(), n
        pick.append(idx)
        n = check_oracle(shard["P"], shard["h_codes"], offs, shard["h_rec"], np.concatenate(pick),
                         "bench shard: 2^31 / 2^32 boundaries, last proteins, long path, published sample")
        assert n >= bench.DUMP_PROTEINS

    def test_long_path_past_2_32(self, shard):
        """Threshold 2048: about 10 000 proteins on the cluster kernels, hundreds of them past residue 2^32."""
        import torch

        nprot, ntotal, offs, lens = self.NPROT, shard["ntotal"], shard["h_offs"], shard["lens"]
        sc = plaac_b200.Scorer(device=0)
        sc.set_long_path(2048)
        out = torch.empty_like(shard["d_rec"])
        n0 = sc.stats().long_proteins
        sc.score_device(shard["d_codes"].data_ptr(), shard["d_offsets"].data_ptr(), nprot, ntotal, out.data_ptr(), sync=True)
        nlong = sc.stats().long_proteins - n0
        sc.close()
        is_long = lens >= 2048
        assert nlong == int(is_long.sum()) > 5_000
        assert int((is_long & (offs[:-1] >= 2**32)).sum()) > 100
        if not torch.equal(out, shard["d_rec"]):
            bad = np.nonzero((rows(device_records(out, nprot)) != rows(shard["h_rec"])).any(axis=1))[0]
            raise AssertionError(f"long path 2048: {len(bad)} records differ from the timed call's, first "
                                 f"{[(int(i), int(lens[i]), int(offs[i])) for i in bad[:10]]} (protein, length, offset)")
        del out
        torch.cuda.empty_cache()
        past = np.nonzero(is_long & (offs[:-1] >= 2**31))[0]
        assert len(past) > 0
        check_oracle(shard["P"], shard["h_codes"], offs, shard["h_rec"], past, "long path 2048, proteins past 2^31")

    def test_host_entry_points_give_the_device_records(self, shard):
        """Scorer.score from pageable memory (about 35 chunks, each rebased) at the automatic long-path threshold, which
        sends the longest proteins of every chunk to the long path; score_packed on 6.3e8 words, and the ranked CORE
        hits of score_packed and score_hits."""
        nprot, ntotal = self.NPROT, shard["ntotal"]
        codes, offs, want = shard["h_codes"], shard["h_offs"], shard["h_rec"]
        sc = plaac_b200.Scorer(device=0)
        try:
            sc.set_long_path(-1)
            got = sc.score(codes, offs)
            n_long = sc.stats().long_proteins
            assert n_long > 1000, n_long
            print(f"host call, automatic threshold: {n_long} proteins on the long path")
            assert_same_records(got, want, "Scorer.score, pageable host memory, automatic long-path threshold")
            del got
            sc.set_long_path(8192)
            words = plaac_b200.pack_words(codes)
            assert len(words) == plaac_b200.lib().plaac_packed_words(ntotal) > 2**29
            lengths = shard["lens"].astype(np.int32)
            got = sc.score_packed(words, lengths, ntotal)
            assert_same_records(got, want, "score_packed")
            del got
            order = self.ranking(shard)
            n_core = int((~np.isnan(want["core_score"])).sum())
            assert n_core > 100_000
            for what in ("score_packed", "score_hits"):
                if what == "score_packed":
                    _, h = sc.score_packed(words, lengths, ntotal, summaries=False, hits="core", capacity=n_core)
                else:
                    h = sc.score_hits(codes, offs, "core", capacity=n_core)
                assert h["n_core"] == n_core and len(h["index"]) == n_core, what
                assert np.array_equal(h["index"], order[:n_core]), what
                assert_same_records(h["records"], want[order[:n_core]], what + " hits")
            del words
        finally:
            sc.close()

    def test_rank_device(self, shard):
        import torch

        nprot = self.NPROT
        d_order = torch.empty(nprot, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        sc = plaac_b200.Scorer(device=0)
        n_core = sc.rank_device(shard["d_rec"].data_ptr(), nprot, d_order.data_ptr())
        sc.close()
        got = d_order.cpu().numpy()
        want = self.ranking(shard)
        assert n_core == int((~np.isnan(shard["h_rec"]["core_score"])).sum())
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, f"rank_device: {len(bad)} positions differ, first {bad[:10].tolist()}"


# ---------------------------------------------------------------------------------------------- 2. a wide batch
@pytest.mark.gpu
class TestWideBatch:
    """17 M short proteins (median 30 residues, 1 to 400): more than 2^24 rows and more than 2^31 bytes of records.
    Many are shorter than the core (LLR -Inf, no CORE), so the ranking has long runs of equal keys."""

    NPROT = 17_000_000
    SEED = 1017

    @pytest.fixture(scope="class")
    def wide(self):
        import torch

        L, dev, n = plaac_b200.lib(), torch.device("cuda", 0), self.NPROT
        lens = torch.empty(n, dtype=torch.int64, device=dev)
        assert L.plaac_bench_synth_lengths(None, self.SEED, 0, n, math.log(30.0), 0.8, 1, 400, lens.data_ptr()) == 0
        offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev)
        torch.cumsum(lens, 0, out=offsets[1:])
        del lens
        ntotal = int(offsets[-1].item())
        codes = torch.empty(ntotal + 64, dtype=torch.uint8, device=dev)
        bg, prd = np.array(bench.BG_SCER, np.float64), np.array(bench.PRD_28, np.float64)
        assert L.plaac_bench_synth_residues(None, self.SEED, 0, n, offsets.data_ptr(), bg.ctypes.data, prd.ctypes.data,
                                            bench.PRD_RATE, bench.X_RATE, codes.data_ptr()) == 0
        recs = torch.empty(n * ROW_BYTES, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        sc = plaac_b200.Scorer(device=0)
        sc.score_device(codes.data_ptr(), offsets.data_ptr(), n, ntotal, recs.data_ptr(), sync=True)
        sc.close()
        d = dict(d_rec=recs, ntotal=ntotal, h_codes=codes[:ntotal].cpu().numpy(), h_offs=offsets.cpu().numpy(),
                 h_rec=device_records(recs, n))
        del codes, offsets, recs
        yield d
        release(d)

    def test_boundaries_and_random_sample_against_oracle(self, wide):
        n, offs, rec = self.NPROT, wide["h_offs"], wide["h_rec"]
        assert n > 2**24 and n * ROW_BYTES > 2**31
        lens = np.diff(offs)
        assert lens.min() >= 1 and lens.max() <= 400 and 20 <= np.median(lens) <= 40
        assert (np.isinf(rec["llr"]).sum() > n // 10) and (~np.isnan(rec["core_score"])).sum() > 1000
        at_2_31_bytes = 2**31 // ROW_BYTES                         # the record that straddles byte 2^31
        pick = [np.arange(max(0, c - BOUNDARY_SPAN), min(n, c + BOUNDARY_SPAN + 1)) for c in (at_2_31_bytes, 2**24)]
        pick.append(np.arange(n - BOUNDARY_SPAN, n))
        pick.append(np.random.default_rng(self.SEED).choice(n, size=RANDOM_SAMPLE, replace=False))
        check_oracle(orc.make_params(), wide["h_codes"], offs, rec, np.concatenate(pick),
                     "17 M proteins: record byte 2^31, row 2^24, last proteins, random sample")

    def test_rank_device_over_all_rows(self, wide):
        import torch

        n = self.NPROT
        d_order = torch.empty(n, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        sc = plaac_b200.Scorer(device=0)
        n_core = sc.rank_device(wide["d_rec"].data_ptr(), n, d_order.data_ptr())
        sc.close()
        got = d_order.cpu().numpy()
        want = web_order(wide["h_rec"])
        assert n_core == int((~np.isnan(wide["h_rec"]["core_score"])).sum())
        bad = np.nonzero(got != want)[0]
        assert len(bad) == 0, f"rank_device, 17 M rows: {len(bad)} positions differ, first {bad[:10].tolist()}"

    def test_host_call_gives_the_device_records(self, wide):
        sc = plaac_b200.Scorer(device=0)
        got = sc.score(wide["h_codes"], wide["h_offs"])
        sc.close()
        assert_same_records(got, wide["h_rec"], "17 M proteins, Scorer.score from host memory")


# ---------------------------------------------------------------------------------------------- 3. FASTA > 2 GiB
def fasta_block(seed=2048, nrec=4000):
    """About 2 MB of FASTA with every quirk of the reader: random \\n / \\r\\n / \\r line ends and line widths, lower
    case, '*' inside and at the end, bytes outside the alphabet, empty records, blank lines followed by text that is
    skipped.  Starts with '>' and ends with a line end."""
    rng = np.random.default_rng(seed)
    alphabet = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYacdxXBZ* 1", dtype=np.uint8)
    parts = []
    for r in range(nrec):
        term = (b"\n", b"\r\n", b"\r")[int(rng.integers(0, 3))]
        parts.append(b">rec%d some text%s" % (r, b"  " if r % 7 == 0 else b"") + term)
        n = int(rng.integers(0, 900))
        seq = alphabet[rng.integers(0, len(alphabet) - (0 if r % 5 == 0 else 3), n)].tobytes()
        if r % 4 == 0:
            seq += b"*"
        w = int(rng.integers(1, 120))
        for k in range(0, len(seq), w):
            parts.append(seq[k:k + w] + term)
        if r % 11 == 0:
            parts.append(term + b"skipped text" + term)
    return b"".join(parts)


def fasta_flags(data):
    """Expected flags of each record: bit 0 the name is trimmed, bit 1 a terminal '*' was stripped."""
    return np.array([(1 if t else 0) | (2 if s.endswith(b"*") else 0) for _, s, t in reference_reader(data)], np.uint8)


@pytest.mark.gpu
class TestFastaPast2GiB:
    TAIL = b">tail record\r\nMKVQQNNQQYQSSGGNQ\r\n>t2\nac*\n"

    @pytest.fixture(scope="class")
    def fasta(self):
        block = fasta_block()
        assert block[:1] == b">" and block[-1:] in (b"\n", b"\r") and len(block) > 1_500_000
        k = (2**31 + 2**20) // len(block) + 1
        text = b"".join([block] * k + [self.TAIL])
        assert len(text) > 2**31 + 2**20 and len(text) % 4096 != 0
        # the expected result of one copy: the first copy starts the file (its first name is trimmed), every later copy
        # reads like the second copy of block + block; the tail like the records after a copy
        names2, codes2, offs2, _ = fasta_expected(block + block)
        flags2 = fasta_flags(block + block)
        nb = (len(names2)) // 2
        nres = int(offs2[nb])
        assert len(names2) == 2 * nb and np.array_equal(codes2[:nres], codes2[nres:])
        names_t, codes_t, offs_t, _ = fasta_expected(block + self.TAIL)
        flags_t = fasta_flags(block + self.TAIL)[nb:]
        counts_b, counts_bt = fasta_expected(block)[3], fasta_expected(block + self.TAIL)[3]
        e = dict(block=block, k=k, nb=nb, nres=nres, codes=codes2[:nres], offs=offs2[:nb + 1],
                 names=(names2[:nb], names2[nb:], names_t[nb:]), flags=(flags2[:nb], flags2[nb:], flags_t),
                 codes_t=codes_t[int(offs_t[nb]):], offs_t=offs_t[nb:] - offs_t[nb],
                 counts=k * counts_b + (counts_bt - counts_b),
                 npos=np.flatnonzero(np.frombuffer(block, np.uint8) == ord(">")) + 1)
        assert len(e["npos"]) == nb
        d = dict(text=text, e=e)
        del text
        yield d
        d.clear()
        gc.collect()

    @staticmethod
    def expected_offsets(e):
        k, nb, nres = e["k"], e["nb"], e["nres"]
        per = (e["offs"][:-1][None, :] + (np.arange(k, dtype=np.int64) * nres)[:, None]).reshape(-1)
        return np.concatenate([per, e["offs_t"] + k * nres])

    def test_ingest(self, fasta):
        text, e = fasta["text"], fasta["e"]
        assert len(text) > 2**31
        k, nb, nres = e["k"], e["nb"], e["nres"]
        nt = len(e["names"][2])
        sc = plaac_b200.Scorer(device=0)
        got = sc.ingest_fasta(text, bg_counts=True)
        sc.close()
        assert len(got["names"]) == k * nb + nt
        assert got["names"] == e["names"][0] + e["names"][1] * (k - 1) + e["names"][2]
        assert np.array_equal(got["offsets"], self.expected_offsets(e))
        codes = got["codes"]
        assert len(codes) == k * nres + len(e["codes_t"])
        for j in range(k):
            assert np.array_equal(codes[j * nres:(j + 1) * nres], e["codes"]), f"codes of copy {j}"
        assert np.array_equal(codes[k * nres:], e["codes_t"])
        want_flags = np.concatenate([e["flags"][0], np.tile(e["flags"][1], k - 1), e["flags"][2]])
        assert np.array_equal(got["flags"], want_flags)
        assert got["bg_counts"].tolist() == e["counts"].tolist()

    def test_score_fasta(self, fasta):
        text, e = fasta["text"], fasta["e"]
        k, nb, nres, block = e["k"], e["nb"], e["nres"], e["block"]
        nrec = k * nb + len(e["names"][2])
        rec = np.zeros(nrec, plaac_b200.SUMMARY_DTYPE)
        offs = np.zeros(nrec + 1, np.int64)
        npos = np.zeros(nrec, np.int64)
        nlen = np.zeros(nrec, np.int32)
        flags = np.zeros(nrec + 8, np.uint8)
        bg = np.zeros(22, np.float64)
        idx = plaac_b200.capi.FastaIndex()
        sc = plaac_b200.Scorer(device=0)
        buf = np.frombuffer(text, np.uint8)
        rc = plaac_b200.lib().plaac_score_fasta(sc._h, buf.ctypes.data, len(text), nrec, rec.ctypes.data, None,
                                                offs.ctypes.data, npos.ctypes.data, nlen.ctypes.data, flags.ctypes.data,
                                                C.byref(idx), bg.ctypes.data)
        assert rc == 0, plaac_b200.lib().plaac_last_error(sc._h).decode()
        first = sc.score(e["codes"], e["offs"])
        sc.close()
        assert idx.nrec == nrec and idx.nres == k * nres + len(e["codes_t"])
        assert np.array_equal(offs, self.expected_offsets(e))
        want_npos = np.concatenate([(e["npos"][None, :] + (np.arange(k, dtype=np.int64) * len(block))[:, None]).reshape(-1),
                                    np.flatnonzero(np.frombuffer(self.TAIL, np.uint8) == ord(">")) + 1 + k * len(block)])
        assert want_npos[-1] > 2**31 and np.array_equal(npos, want_npos)
        assert np.array_equal(nlen[nb:k * nb], np.tile(nlen[:nb], k - 1))
        assert bg.tolist() == e["counts"].tolist()
        assert_same_records(rec[:nb], first, "plaac_score_fasta, first copy vs Scorer.score")
        r = rows(rec)
        for j in range(1, k):
            bad = np.nonzero((r[j * nb:(j + 1) * nb] != r[:nb]).any(axis=1))[0]
            assert len(bad) == 0, f"copy {j} (text offset {j * len(block)}): records {bad[:10].tolist()} differ from copy 0"


# ---------------------------------------------------------------------------------------------- 4. variants
@pytest.mark.gpu
def test_saturation_scan_past_2_32_residues():
    """Every substitution of one 34 000-residue protein: 646 001 variants, 2.2e10 residues in one call."""
    codes, offs = synth.long_proteins(seed=2001, lengths=(34000,))
    protein, first_sub, pos, code = var = plaac_b200.saturation(codes, offs)
    nvar = len(protein)
    vres = int(np.diff(offs)[protein].sum())
    assert vres > 2**32 and nvar == 1 + 34000 * 19 + int((codes == 0).sum() + (codes == 21).sum())
    sc = plaac_b200.Scorer(device=0)
    try:
        rec = sc.score_variants(codes, offs, *var)
        eff, wild = sc.variant_effects(codes, offs, *var, columns=plaac_b200.EFFECT_COLUMNS, wild=True)
        assert wild.tobytes() == sc.score(codes, offs).tobytes()
        rng = np.random.default_rng(34000)
        pick = np.unique(np.concatenate([np.arange(500), np.arange(nvar - 500, nvar),
                                         rng.choice(nvar, size=2000, replace=False)]))
        sub_first = np.concatenate([[0], np.cumsum(first_sub[pick + 1] - first_sub[pick])])
        sub_at = np.concatenate([np.arange(first_sub[v], first_sub[v + 1]) for v in pick]).astype(np.int64)
        mc, mo = materialise(codes, offs, protein[pick], sub_first, pos[sub_at], code[sub_at])
        want = sc.score(mc, mo)
    finally:
        sc.close()
    assert_same_bytes(rec[pick], want, "variant records vs the materialised variants")
    P = orc.make_params()
    ref = orc.score_batch(P, mc, mo, nthreads=NT)
    _check(rec[pick], ref, f"saturation scan, {len(pick)} variants", P, mc, mo, max_ties=1 + len(pick) // 20_000)
    # effects: record minus wild type, bit for bit, over the whole call (NaN equal to NaN)
    assert_same_effects(eff, effects_expected(rec, wild, protein, plaac_b200.EFFECT_COLUMNS), "effects, all variants")
    has = lambda r: (r["core_start"] >= 0).astype(np.float64)  # noqa: E731
    assert np.array_equal(eff["core_change"], has(rec) - has(wild[protein]))
