"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Integers bit-exact, doubles within 1e-9 relative (tests/parity.py states the exact rule)."""
import json
import math
import os

import numpy as np
import pytest

import plaac_b200
from oracle import orc
from tests import parity, synth

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NT = max(1, min(32, os.cpu_count() or 1))


@pytest.fixture(scope="module")
def scorer():
    s = plaac_b200.Scorer(device=0)
    yield s
    s.close()


def _check(got, ref, what="", P=None, codes=None, offs=None, max_ties=0, reassociated=()):
    if P is not None:
        bad, nties = parity.compare_with_tie_classes(P, codes, offs, got, ref, orc.INT_FIELDS, orc.DBL_FIELDS)
        assert nties <= max_ties, f"{what}: {nties} PAPA tie-class rows (allowed {max_ties})"
    else:
        bad = parity.compare_summaries(got, ref, orc.INT_FIELDS, orc.DBL_FIELDS)
    assert not bad, what + "\n" + "\n".join(bad[:40])
    # columns evaluated in reference operation order must be (nearly) bit-exact, far inside the 1e-9 bar
    for f in parity.REF_ORDER:
        if f == "papa_llr" and P is not None:
            continue  # follows the centre; covered by the tie-class rule
        if f in reassociated:
            continue  # long-sequence path: chunk-wise sums, held to the 1e-9 bar only
        assert parity.max_rel(got, ref, f) <= 1e-13, (what, f, parity.max_rel(got, ref, f))


def test_classic_prions_against_golden_fixture(scorer, golden):
    seqs = [plaac_b200.encode(p["seq"]) for p in golden["proteins"]]
    codes, offs = plaac_b200.pack(seqs)
    got = scorer.score(codes, offs)
    for i, prot in enumerate(golden["proteins"]):
        for k, v in prot["summary"].items():
            if isinstance(v, int):
                assert int(got[i][k]) == v, (prot["name"], k)
            elif math.isnan(v):
                assert math.isnan(got[i][k])
            else:
                assert parity.close(got[i][k], v, parity.SCALE[k]), (prot["name"], k, got[i][k], v)
    _check(got, orc.score_batch(orc.make_params(), codes, offs), "classic prions")


def test_encode_matches_reference_alphabet():
    s = "XACDEFGHIKLMNPQRSTVWY*acdefghiklmnpqrstvwyxBJOUZ -1\t"
    assert list(plaac_b200.encode(s, strip_stop=False)) == list(orc.encode(s, strip_stop=False))
    assert list(plaac_b200.encode("MKV*")) == [11, 9, 18]


def test_edge_cases(scorer):
    codes, offs = synth.edge_cases()
    got = scorer.score(codes, offs)
    P = orc.make_params()
    ref = orc.score_batch(P, codes, offs)
    # poly-Q / poly-P plateaus: the jar's PAPAcen is decided by its own rounding noise (tie class)
    _check(got, ref, "edge cases", P, codes, offs, max_ties=4)
    assert (got["prot_len"] == np.diff(offs)).all()


def test_empty_and_zero_length_inputs(scorer):
    assert len(scorer.score(np.zeros(0, np.uint8), np.zeros(1, np.int64))) == 0
    codes, offs = plaac_b200.pack([np.array([12, 14, 12], np.uint8), np.zeros(0, np.uint8), np.array([1], np.uint8)])
    got = scorer.score(codes, offs)
    ref = orc.score_batch(orc.make_params(), codes, offs)
    assert got["prot_len"].tolist() == [3, 0, 1]
    _check(got[[0, 2]], ref[[0, 2]], "around an empty record")


def test_yeast_sized_proteome(scorer):
    """Config 2 size (about 6k proteins / 3M residues), default parameters."""
    codes, offs = synth.proteome(6000, seed=1001)
    got = scorer.score(codes, offs)
    ref = orc.score_batch(orc.make_params(), codes, offs, nthreads=NT)
    _check(got, ref, "yeast-sized")
    assert (ref["core_start"] >= 0).sum() > 100  # the injected Q/N-rich segments are found


def test_human_sized_blended_background(scorer):
    """Config 3: human-like lengths, alpha = 0.5 blend of yeast and human backgrounds."""
    kw = dict(alpha=0.5, bg_counts=synth.BG_HUMAN_COUNTS)
    bg = synth.BG_HUMAN_COUNTS.copy()
    bg[0] = 0
    codes, offs = synth.proteome(20000, seed=1002, median=415.0, sigma=0.75, bg=bg)
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    got = sc.score(codes, offs)
    sc.close()
    ref = orc.score_batch(orc.make_params(**kw), codes, offs, nthreads=NT)
    _check(got, ref, "human-sized")


def test_long_sequences(scorer):
    """Config 5: 35k and 100k residues, through the chunked long-sequence path (scan of 2x2 max-plus matrices for
    Viterbi, warm-started chunks for the LUT forward recurrence) and, with the path switched off, through the bucketed
    kernel in plaac.java's own operation order."""
    codes, offs = synth.long_proteins()
    ref = orc.score_batch(orc.make_params(), codes, offs, nthreads=2)
    before = scorer.stats().long_proteins
    got = scorer.score(codes, offs)
    assert scorer.stats().long_proteins == before + 2
    _check(got, ref, "long sequences (long path)")
    print("forward chunks redone:", scorer.stats().long_redone_chunks)
    assert (got["core_start"] >= 0).all()
    scorer.set_long_path(0)
    try:
        got = scorer.score(codes, offs)
        assert scorer.stats().long_proteins == before + 2
        _check(got, ref, "long sequences (bucketed kernel)")
    finally:
        scorer.set_long_path(8192)


def test_long_path_mixed_batch_thresholds_and_fallback():
    """Proteins on both sides of the threshold in one batch (host and device-resident API), lengths around the chunk
    geometry, the sequential-forward fallback, and a warm-up too short to forget its start (must be detected)."""
    rng = np.random.default_rng(77)
    bg = synth.BG_SCER / synth.BG_SCER.sum()
    prd = synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for n in (1023, 1024, 1025, 2047, 2048, 4095, 4096, 4097, 8191, 8192, 8193, 12287, 12288, 12289, 20000, 98303, 98304,
              98305):
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        for frac in (0.0, 0.31, 0.77):
            st = int(n * frac)
            if rng.random() < 0.7:
                s[st:st + 120] = rng.choice(22, size=min(120, n - st), p=prd)
        if n % 2:
            s[-200:] = rng.choice(22, size=200, p=prd)  # PrD reaching the last residue
        seqs.append(s)
    seqs.append(np.full(5000, 14, np.uint8))                                    # poly-Q: plateaus, one Viterbi run
    seqs.append(np.tile(np.array([13, 1, 13, 13, 12], np.uint8), 1200))        # proline rule across chunk borders
    seqs.append(rng.integers(1, 21, size=6000).astype(np.uint8))               # uniform composition
    c2, o2 = synth.proteome(800, seed=5)
    seqs += [c2[o2[i]:o2[i + 1]] for i in range(800)]
    order = rng.permutation(len(seqs))
    seqs = [seqs[i] for i in order]
    codes, offs = plaac_b200.pack(seqs)
    P = orc.make_params()
    ref = orc.score_batch(P, codes, offs, nthreads=NT)
    lens = np.diff(offs)
    redone = {}
    for min_len, warm in [(1024, 0), (4096, 0), (1024, -1), (1024, 3)]:
        sc = plaac_b200.Scorer(device=0)
        sc.set_long_path(min_len, warm)
        got = sc.score(codes, offs)
        st = sc.stats()
        assert st.long_proteins == int((lens >= min_len).sum())
        redone[(min_len, warm)] = st.long_redone_chunks
        _check(got, ref, f"long path min_len={min_len} warm={warm}", P, codes, offs, max_ties=2)
        sc.close()
    print("forward chunks redone:", redone)
    # a 3-residue warm-up cannot forget its start: the entry test must catch (nearly) every chunk
    assert redone[(1024, 3)] > 10 * max(1, redone[(1024, 0)])
    # device-resident API (the long list is selected and sized on the device)
    import torch

    sc = plaac_b200.Scorer(device=0)
    sc.set_long_path(2048)
    d_codes = torch.from_numpy(codes).cuda()
    d_offs = torch.from_numpy(offs).cuda()
    d_out = torch.zeros((len(lens), 160), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    sc.score_device(d_codes.data_ptr(), d_offs.data_ptr(), len(lens), int(offs[-1]), d_out.data_ptr())
    got = d_out.cpu().numpy().reshape(-1).view(plaac_b200.SUMMARY_DTYPE)
    assert sc.stats().long_proteins == int((lens >= 2048).sum())
    _check(got, ref, "long path, device API", P, codes, offs, max_ties=2)
    sc.close()


def test_long_path_around_the_chunk_geometry():
    """Long proteins of 8 192 to 60 001 residues on the default path (two CTAs of k_long_score per protein beside the
    cluster kernel), some ending exactly on a chunk boundary (8 192 and 49 152: 32 and 192 chunks of 256 residues) and
    others one residue off it or between, with Q/N-rich segments at a seventh, the middle and the end: records must be
    right."""
    rng = np.random.default_rng(4242)
    bg = synth.BG_SCER / synth.BG_SCER.sum()
    prd = synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for n in (8192, 9001, 24577, 49151, 49152, 60001):
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        for st in (n // 7, n // 2, n - 150):
            s[st:st + 150] = rng.choice(22, size=150, p=prd)
        seqs.append(s)
    codes, offs = plaac_b200.pack(seqs)
    ref = orc.score_batch(orc.make_params(), codes, offs, nthreads=NT)
    sc = plaac_b200.Scorer(device=0)
    got = sc.score(codes, offs)
    assert sc.stats().long_proteins == len(seqs)
    sc.close()
    _check(got, ref, "long path around the chunk geometry")


@pytest.mark.parametrize("kw", [dict(core_len=30), dict(core_len=100, ww1=21, ww2=21), dict(ww1=40, ww2=40),
                                dict(adjust_prolines=False), dict(core_len=7, ww1=5, ww2=5), dict(ww1=1, ww2=1),
                                # -w and -W with different half-widths: the tap-by-tap kernels of generic_windows.cuh
                                dict(ww1=31, ww2=51), dict(ww1=52, ww2=9, core_len=30), dict(ww1=41, ww2=40),
                                dict(ww1=3, ww2=120, adjust_prolines=False),
                                # windows longer than most proteins (look-back beyond the residue rings)
                                dict(ww1=601, ww2=601), dict(ww1=2000, ww2=41, core_len=90),
                                # a core length beyond the throughput kernel's rings: reference-order anchor kernel
                                dict(core_len=1500)])
def test_other_parameters(kw):
    codes, offs = synth.proteome(1500, seed=11, median=200.0)
    e, eo = synth.edge_cases()
    codes, offs = np.concatenate([codes, e]), np.concatenate([offs, eo[1:] + offs[-1]])
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    got = sc.score(codes, offs)
    sc.close()
    P = orc.make_params(**kw)
    ref = orc.score_batch(P, codes, offs, nthreads=NT)
    _check(got, ref, str(kw), P, codes, offs, max_ties=6)


def _composition_ties(codes, offs, starts, width=60):
    """(proteins whose chosen window has a composition-identical twin, those where the choice is not the earliest twin)"""
    tied = later = 0
    for i in range(len(offs) - 1):
        s, st = codes[offs[i]:offs[i + 1]], int(starts[i])
        if st < 0:
            continue
        cum = np.zeros((len(s) + 1, 22), np.int32)
        cum[np.arange(1, len(s) + 1), s] = 1
        cum = cum.cumsum(0)
        comp = cum[width:] - cum[:-width]
        twins = np.nonzero((comp == comp[st]).all(1))[0]
        tied += len(twins) > 1
        later += bool(twins[0] < st)
    return tied, later


def test_composition_identical_best_windows(scorer):
    """Proteins with repeated Q/N-rich blocks (tests/synth.py repeat_proteome): many have several best LLR and CORE
    windows of identical composition, and the reference picks the one its running sums round highest -- often not the
    earliest, and for the CORE over sums polluted by the -1e6 mask.  LLR and CORE positions and scores must match the
    oracle exactly.  A copied block can also put two PAPA centres on a plateau equal to the last bit: the PAPA fields
    are held to the documented tie-class rule, for at most two proteins."""
    codes, offs = synth.repeat_proteome(1500, seed=2024)
    got = scorer.score(codes, offs)
    P = orc.make_params()
    ref = orc.score_batch(P, codes, offs, nthreads=NT)
    _check(got, ref, "composition-identical best windows", P, codes, offs, max_ties=2)
    for f in ("llr_start", "core_start"):
        tied, later = _composition_ties(codes, offs, ref[f])
        assert tied > 300 and later > 100, (f, tied, later)


def test_chunked_host_path_and_permutation_invariance(scorer):
    """Results are per-protein: independent of batch composition, order and chunking."""
    codes, offs = synth.proteome(3000, seed=5, median=300.0)
    full = scorer.score(codes, offs)
    sc = plaac_b200.Scorer()
    sc.set_chunk(max_residues=50_000, max_proteins=257)
    chunked = sc.score(codes, offs)
    sc.close()
    assert full.tobytes() == chunked.tobytes()
    rng = np.random.default_rng(0)
    perm = rng.permutation(len(offs) - 1)
    pc, po = plaac_b200.pack([codes[offs[i]:offs[i + 1]] for i in perm])
    shuffled = scorer.score(pc, po)
    assert shuffled.tobytes() == full[perm].tobytes()


def test_invalid_inputs_are_reported(scorer):
    with pytest.raises(plaac_b200.PlaacError) as e:
        scorer.score(np.array([1, 2, 40, 3], np.uint8), np.array([0, 4], np.int64))
    assert e.value.code == -1
    with pytest.raises(plaac_b200.PlaacError) as e:
        scorer.score(np.array([1, 2, 3], np.uint8), np.array([0, 2, 1], np.int64))
    assert e.value.code == -1
    with pytest.raises(plaac_b200.PlaacError) as e:
        plaac_b200.Scorer(plaac_b200.default_params(ww1=0, ww2=21))
    assert e.value.code == -1
    # -w / -W with different half-widths used to be PLAAC_E_UNSUPPORTED: now scored (generic_windows.cuh)
    plaac_b200.Scorer(plaac_b200.default_params(ww1=41, ww2=21)).close()
    # the ctx still works afterwards
    got = scorer.score(np.array([1, 2, 3], np.uint8), np.array([0, 3], np.int64))
    assert got["prot_len"][0] == 3
    # an invalid code inside a LONG protein in per-residue mode without records (only k_long_post sees its residues):
    # scored as X, reported after the batch
    import torch
    rng = np.random.default_rng(3)
    seq = rng.integers(1, 21, size=3000).astype(np.uint8)
    seq[1234] = 77
    sc = plaac_b200.Scorer()
    sc.set_long_path(1024)
    dc = torch.from_numpy(np.concatenate([seq, np.zeros(64, np.uint8)])).cuda()
    do = torch.tensor([0, 3000], dtype=torch.int64, device="cuda")
    u8 = torch.zeros(2 * 3000, dtype=torch.uint8, device="cuda")
    f64 = torch.zeros(10 * 3000, dtype=torch.float64, device="cuda")
    ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + 3000}
    for k, nm in enumerate(plaac_b200.RESIDUE_F64):
        ptrs[nm] = f64.data_ptr() + 8 * k * 3000
    with pytest.raises(plaac_b200.PlaacError) as e:
        sc.score_device(dc.data_ptr(), do.data_ptr(), 1, 3000, 0, residue_ptrs=ptrs, sync=True)
    assert e.value.code == -1
    seq[1234] = 0
    ref = orc.residue_batch(orc.make_params(), seq, np.array([0, 3000], np.int64))
    assert (u8.cpu().numpy()[3000:] == ref["map"]).all()
    assert np.abs(f64.cpu().numpy()[9 * 3000:] - ref["post_prd"]).max() < 1e-9
    sc.close()


def test_pinned_host_buffers(scorer):
    """plaac_host_alloc (plain and write-combined) and plaac_host_register: same records as from pageable memory."""
    codes, offs = synth.proteome(3000, seed=11)
    n = len(offs) - 1
    ref = scorer.score(codes, offs)
    with plaac_b200.PinnedBuffer(len(codes), np.uint8, write_combined=True) as pc, \
            plaac_b200.PinnedBuffer(len(offs), np.int64) as po, \
            plaac_b200.PinnedBuffer(n, plaac_b200.SUMMARY_DTYPE) as ps:
        pc.array[:] = codes
        po.array[:] = offs
        scorer.score_ptr(pc.ptr, po.ptr, n, ps.ptr)
        assert ps.array.tobytes() == ref.tobytes()
    c2 = codes.copy()
    plaac_b200.host_register(c2)
    try:
        assert scorer.score(c2, offs).tobytes() == ref.tobytes()
    finally:
        plaac_b200.host_unregister(c2)
    with pytest.raises(plaac_b200.PlaacError):
        plaac_b200.host_unregister(np.zeros(64, np.uint8))  # never registered
    with pytest.raises(plaac_b200.PlaacError):
        plaac_b200.host_register(np.zeros(0, np.uint8))


def test_device_resident_api_and_stats(scorer):
    import torch

    codes, offs = synth.proteome(2000, seed=9)
    ref = scorer.score(codes, offs)
    dc = torch.from_numpy(codes).cuda()
    do = torch.from_numpy(offs).cuda()
    out = torch.zeros(len(offs) - 1, 160, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    before = scorer.stats().kernel_launches
    scorer.score_device(dc.data_ptr(), do.data_ptr(), len(offs) - 1, int(offs[-1]), out.data_ptr())
    got = out.cpu().numpy().view(plaac_b200.SUMMARY_DTYPE).reshape(-1)
    assert got.tobytes() == ref.tobytes()
    st = scorer.stats()
    assert 7 <= st.kernel_launches - before <= 11 and st.last_score_ms > 0 and st.last_total_ms >= st.last_score_ms


def test_throughput_kernel_against_reference_order_anchor_at_scale():
    """v2 (role-split, running sums) vs v1 (single fused kernel in plaac.java's operation order) on a set far
    larger than the CPU oracle can check quickly: integers identical, reference-order columns bit-identical."""
    codes, offs = synth.proteome(150_000, seed=77, median=290.0, sigma=0.62)
    a = plaac_b200.Scorer()
    a.set_kernel_variant(1)
    b = plaac_b200.Scorer()
    b.set_kernel_variant(2)
    ra, rb = a.score(codes, offs), b.score(codes, offs)
    a.close()
    b.close()
    same_cen = ra["papa_center"] == rb["papa_center"]
    assert same_cen.mean() > 0.9999
    for f in orc.INT_FIELDS:
        if f != "papa_center":
            assert (ra[f] == rb[f]).all(), f
    for f in ("llr", "core_score", "prd_score", "hmm_all", "hmm_vit", "fi_meanhydro", "fi_meancharge", "fi_meancombo"):
        assert ra[f].tobytes() == rb[f].tobytes(), f
    for f in ("papa_prop", "papa_fi", "papa_llr", "papa_llr2", "papa_combo"):
        assert parity.close(rb[f][same_cen], ra[f][same_cen], parity.SCALE[f]).all(), f


def test_throughput_kernels_v2_and_v3_give_the_same_bytes():
    """Variant 3 (default: packed Q/N window counting, roles mixed over the scheduler partitions) is variant 2's
    arithmetic with fewer instructions: every byte of every record is the same, also with a long core / wide MW window
    where the packed counting is switched off."""
    codes, offs = synth.proteome(150_000, seed=78, median=290.0, sigma=0.62)
    for params in (None, plaac_b200.default_params(core_len=100, ww1=61, ww2=61)):
        a = plaac_b200.Scorer(params)
        a.set_kernel_variant(2)
        b = plaac_b200.Scorer(params)
        b.set_kernel_variant(3)
        c = plaac_b200.Scorer(params)
        ra, rb, rc = a.score(codes, offs), b.score(codes, offs), c.score(codes, offs)
        for s in (a, b, c):
            s.close()
        assert ra.tobytes() == rb.tobytes() == rc.tobytes()


# ----------------------------------------------------------------------------- per-residue mode (config 2)
def _check_residue(got, ref, what=""):
    for k in orc.RESIDUE_U8:
        bad = np.nonzero(got[k] != ref[k])[0]
        assert len(bad) == 0, (what, k, len(bad), bad[:5])
    for k in orc.RESIDUE_F64:
        assert (np.isnan(got[k]) == np.isnan(ref[k])).all(), (what, k, "NaN pattern")
        ok = parity.close(got[k], ref[k], parity.SCALE[k])
        assert ok.all(), (what, k, int((~ok).sum()), got[k][~ok][:3], ref[k][~ok][:3])


def test_per_residue_against_golden_fixture(scorer, golden):
    seqs = [plaac_b200.encode(p["seq"]) for p in golden["proteins"]]
    codes, offs = plaac_b200.pack(seqs)
    summ, res = scorer.score(codes, offs, per_residue=True)
    for i, prot in enumerate(golden["proteins"]):
        lo = int(offs[i])
        for k, vals in prot["residue"].items():
            for j, v in zip(prot["residue_idx"], vals):
                x = res[k][lo + j]
                if v is None:
                    assert x != x, (prot["name"], k, j)
                elif k in orc.RESIDUE_U8:
                    assert int(x) == int(v), (prot["name"], k, j)
                else:
                    assert parity.close(x, v, parity.SCALE[k]), (prot["name"], k, j, x, v)
        runs = lambda bits: [[int(a), int(b)] for a, b in zip(
            np.nonzero(np.diff(np.r_[0, bits.astype(np.int64), 0]) == 1)[0],
            np.nonzero(np.diff(np.r_[0, bits.astype(np.int64), 0]) == -1)[0] - 1)]
        assert runs(res["vit"][lo:int(offs[i + 1])]) == prot["vit_runs"]
        assert runs(res["map"][lo:int(offs[i + 1])]) == prot["map_runs"]
    # the summary rows of the same call are the summary-mode rows
    assert summ.tobytes() == scorer.score(codes, offs).tobytes()


def test_per_residue_yeast_sized(scorer):
    """Config 2: yeast-proteome-sized set with per-residue Viterbi parse and posterior output."""
    codes, offs = synth.proteome(6000, seed=1001)
    _, got = scorer.score(codes, offs, per_residue=True)
    ref = orc.residue_batch(orc.make_params(), codes, offs, nthreads=NT)
    _check_residue(got, ref, "yeast-sized per-residue")


def test_per_residue_edge_cases_and_chunking():
    codes, offs = synth.edge_cases()
    sc = plaac_b200.Scorer()
    sc.set_chunk(max_residues=3000, max_proteins=7)
    _, got = sc.score(codes, offs, per_residue=True)
    sc.close()
    ref = orc.residue_batch(orc.make_params(), codes, offs)
    _check_residue(got, ref, "edge cases per-residue")


@pytest.mark.parametrize("kw", [dict(ww1=31, ww2=51), dict(ww1=52, ww2=9, alpha=0.5)])
def test_per_residue_windows_with_different_half_widths(kw):
    """-w / -W independent (generic_windows.cuh): per-residue tracks and the summary records of the same call, host API
    in several chunks and device-resident API."""
    codes, offs = synth.proteome(700, seed=31, median=180.0)
    e, eo = synth.edge_cases()
    codes, offs = np.concatenate([codes, e]), np.concatenate([offs, eo[1:] + offs[-1]])
    # ... and two long proteins: with the threshold below they take the long-sequence paths (records: k_long_score,
    # posteriors / MAP: k_long_post) while every window column still comes from the tap-by-tap kernels
    lc, lo = synth.long_proteins(seed=4, lengths=(2500, 6000))
    codes, offs = np.concatenate([codes, lc]), np.concatenate([offs, lo[1:] + offs[-1]])
    P = orc.make_params(**kw)
    ref_s = orc.score_batch(P, codes, offs, nthreads=NT)
    ref_r = orc.residue_batch(P, codes, offs)
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    sc.set_chunk(40000, 300)
    sc.set_long_path(2048)
    got_s, got_r = sc.score(codes, offs, per_residue=True)
    sc.close()
    _check(got_s, ref_s, f"summary beside per-residue {kw}", P, codes, offs, max_ties=6)
    _check_residue(got_r, ref_r, f"per-residue {kw}")
    # the window tracks are evaluated tap by tap in the jar's order: the same bits as the oracle's
    for k in ("hydro", "charge", "fi", "plaac", "papa", "fix2", "plaacx2", "papax2"):
        a, b = got_r[k], ref_r[k]
        assert ((a == b) | (np.isnan(a) & np.isnan(b))).all(), k


@pytest.mark.parametrize("plus,minus", [((3, 4, 7), (9, 15, 2)), ((3, 20), (9,)), ((), (15,)), ((4, 5), (3,))])
def test_other_charge_classes(plus, minus):
    """aacharge tables other than PLAAC's (:37-60): k_pack's general class tests (sets of any size, a +1 set that is
    not a run of consecutive codes, an empty set) against the oracle, records and per-residue tracks."""
    codes, offs = synth.proteome(600, seed=77, median=150.0)
    e, eo = synth.edge_cases()
    codes, offs = np.concatenate([codes, e]), np.concatenate([offs, eo[1:] + offs[-1]])
    P = orc.make_params()
    gp = plaac_b200.default_params()
    for i in range(len(P.charge)):
        c = 1.0 if i in plus else (-1.0 if i in minus else 0.0)
        P.charge[i] = c
        gp.charge[i] = c
    ref_s = orc.score_batch(P, codes, offs, nthreads=NT)
    ref_r = orc.residue_batch(P, codes, offs)
    sc = plaac_b200.Scorer(gp)
    got_s, got_r = sc.score(codes, offs, per_residue=True)
    only_s = sc.score(codes, offs)
    sc.close()
    _check(got_s, ref_s, f"charge classes +{plus} -{minus}", P, codes, offs, max_ties=6)
    _check(only_s, ref_s, f"charge classes +{plus} -{minus} (records only)", P, codes, offs, max_ties=6)
    _check_residue(got_r, ref_r, f"charge classes +{plus} -{minus}")


def test_per_residue_long_and_other_params():
    codes, offs = synth.long_proteins(lengths=(35000,))
    kw = dict(core_len=30, ww1=21, ww2=21, alpha=0.5, bg_counts=synth.BG_HUMAN_COUNTS)
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    _, got = sc.score(codes, offs, per_residue=True)
    sc.close()
    ref = orc.residue_batch(orc.make_params(**kw), codes, offs)
    _check_residue(got, ref, "long per-residue")


def _residue_equal_bits(a, b, what):
    for k in orc.RESIDUE_U8:
        assert (a[k] == b[k]).all(), (what, k, int((a[k] != b[k]).sum()))
    for k in orc.RESIDUE_F64:
        same = (a[k] == b[k]) | (np.isnan(a[k]) & np.isnan(b[k]))
        assert same.all(), (what, k, int((~same).sum()), a[k][~same][:3], b[k][~same][:3])


def test_per_residue_long_path_matches_the_sequential_walk_bit_for_bit(monkeypatch):
    """Long proteins in per-residue mode (long_residue.cuh: one thread-block cluster per protein, binade-frame forward
    and backward recurrences with an exact carry over the chunk boundaries) against (i) the oracle and (ii) the bucketed
    kernels' single-lane walk of the same proteins: the same bits in every column, in both cluster size classes, with
    several warm-up lengths (3 residues: most chunks are redone sequentially), mixed with short proteins, with and
    without records in the same call, through the host API and the device-resident one."""
    rng = np.random.default_rng(77)
    lc, lo = synth.long_proteins(seed=1009, lengths=(1300, 9000, 35000, 2049, 100000))
    sc_, so = synth.proteome(300, seed=5, median=300.0)
    codes = np.concatenate([sc_[:so[150]], lc, sc_[so[150]:]])
    lens = np.concatenate([np.diff(so)[:150], np.diff(lo), np.diff(so)[150:]])
    offs = np.zeros(len(lens) + 1, np.int64)
    np.cumsum(lens, out=offs[1:])
    P = orc.make_params()
    ref = orc.residue_batch(P, codes, offs, nthreads=NT)
    ref_s = orc.score_batch(P, codes, offs, nthreads=NT)

    sc = plaac_b200.Scorer()
    sc.set_long_path(0)
    _, walk = sc.score(codes, offs, per_residue=True)
    assert sc.stats().long_proteins == 0
    sc.close()
    _check_residue(walk, ref, "sequential walk")

    import torch
    dev = torch.device("cuda", 0)
    dc = torch.from_numpy(np.concatenate([codes, np.zeros(64, np.uint8)])).to(dev)
    do = torch.from_numpy(offs).to(dev)
    ntot = int(offs[-1])
    u8 = torch.zeros(2 * ntot, dtype=torch.uint8, device=dev)
    f64 = torch.zeros(10 * ntot, dtype=torch.float64, device=dev)
    ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + ntot}
    for k, nm in enumerate(plaac_b200.RESIDUE_F64):
        ptrs[nm] = f64.data_ptr() + 8 * k * ntot

    def device_call(sc, what):
        # per-residue arrays only (no records): the Viterbi parse of the long proteins then comes from k_long_post
        u8.zero_()
        f64.zero_()
        sc.score_device(dc.data_ptr(), do.data_ptr(), len(lens), ntot, 0, residue_ptrs=ptrs, sync=True)
        h8, hf = u8.cpu().numpy(), f64.cpu().numpy()
        dev_got = {"vit": h8[:ntot], "map": h8[ntot:]}
        for k, nm in enumerate(plaac_b200.RESIDUE_F64):
            dev_got[nm] = hf[k * ntot:(k + 1) * ntot]
        _residue_equal_bits(dev_got, walk, "device-resident, no records: " + what)

    for warm, big_min, ties in ((256, None, None), (3, None, None), (64, "1024", None), (256, "200000", None), (256, None, "1")):
        # (the test hooks are read when the Scorer is created)
        if big_min:
            monkeypatch.setenv("PLAAC_LP_BIG_MIN", big_min)
        if ties:
            monkeypatch.setenv("PLAAC_LONG_TIES", ties)   # every binade a tie binade: every Viterbi chunk redone sequentially
        sc = plaac_b200.Scorer()
        what = f"warm={warm} big_min={big_min} ties={ties}"
        sc.set_long_path(1024, warm)
        summ, got = sc.score(codes, offs, per_residue=True)
        assert sc.stats().long_proteins == int((lens >= 1024).sum())
        _check_residue(got, ref, "long per-residue " + what)
        _residue_equal_bits(got, walk, "long path vs walk " + what)
        _check(summ, ref_s, "records beside the long per-residue path", P, codes, offs, max_ties=2)
        device_call(sc, what)
        sc.close()
        if big_min:
            monkeypatch.delenv("PLAAC_LP_BIG_MIN")
        if ties:
            monkeypatch.delenv("PLAAC_LONG_TIES")
    # automatic threshold
    sc = plaac_b200.Scorer()
    sc.set_long_path(-1, 256)
    _, got = sc.score(codes, offs, per_residue=True)
    assert sc.stats().long_proteins > 0
    _residue_equal_bits(got, walk, "automatic threshold")
    device_call(sc, "automatic threshold")
    sc.close()


def test_many_proteins_on_the_long_paths():
    """A threshold far below what the path is meant for: 500 proteins of 1 030 - 1 400 residues each get their own CTAs
    (scratch proportional to the residues, not to the number of proteins); records and per-residue arrays against the oracle."""
    rng = np.random.default_rng(99)
    lens = rng.integers(1030, 1400, size=500)
    bgp, prdp = synth.BG_SCER / synth.BG_SCER.sum(), synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for i, n in enumerate(lens):
        s = rng.choice(22, size=int(n), p=bgp).astype(np.uint8)
        if i % 3 == 0:
            st = int(rng.integers(0, n - 200))
            s[st:st + 150] = rng.choice(22, size=150, p=prdp)
        seqs.append(s)
    codes, offs = plaac_b200.pack(seqs)
    P = orc.make_params()
    ref_s = orc.score_batch(P, codes, offs, nthreads=NT)
    ref_r = orc.residue_batch(P, codes, offs, nthreads=NT)
    sc = plaac_b200.Scorer()
    sc.set_long_path(1024)
    got_s = sc.score(codes, offs)
    assert sc.stats().long_proteins == 500
    _check(got_s, ref_s, "500 proteins on the long path, records", P, codes, offs, max_ties=3)
    got_s2, got_r = sc.score(codes, offs, per_residue=True)
    sc.close()
    assert got_s2.tobytes() == got_s.tobytes()
    _check_residue(got_r, ref_r, "500 proteins on the long path, per-residue")


@pytest.mark.parametrize("kw", [dict(core_len=100, ww1=21, ww2=21), dict(core_len=7, ww1=5, ww2=5),
                                dict(core_len=30, ww1=40, ww2=40, adjust_prolines=False),
                                dict(alpha=0.5, bg_counts=synth.BG_HUMAN_COUNTS), dict(core_len=250, ww1=61, ww2=61),
                                dict(ww1=31, ww2=51)])
def test_long_path_other_parameters(kw):
    """The chunked long-sequence path with other window / core sizes and a blended background: chunk geometry
    (a chunk holds a whole CORE / MW window), halo widths and the binade-frame passes all depend on them."""
    rng = np.random.default_rng(123)
    bg = synth.BG_SCER / synth.BG_SCER.sum()
    prd = synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for n in (4096, 5001, 7777, 12345, 30011):
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        for frac in (0.05, 0.4, 0.93):
            st = int(n * frac)
            s[st:st + 260] = rng.choice(22, size=min(260, n - st), p=prd)
        seqs.append(s)
    c2, o2 = synth.proteome(300, seed=6)
    seqs += [c2[o2[i]:o2[i + 1]] for i in range(300)]
    codes, offs = plaac_b200.pack(seqs)
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    sc.set_long_path(4096)
    got = sc.score(codes, offs)
    assert sc.stats().long_proteins == 5
    sc.close()
    P = orc.make_params(**kw)
    ref = orc.score_batch(P, codes, offs, nthreads=NT)
    _check(got, ref, "long path " + str(kw), P, codes, offs, max_ties=3)


def test_long_path_automatic_threshold():
    """Automatic threshold (plaac_set_long_path(-1)): at most one wave of CTAs, never below 1024 residues, and only proteins whose
    sequential walk would show in the batch's time -- host-buffer and device-resident API agree with each other, with
    the bucketed kernel."""
    import torch

    codes, offs = synth.proteome(6000, seed=1001)          # yeast-sized: ~8 % of the proteins have >= 1024 residues
    lens = np.diff(offs)
    sc = plaac_b200.Scorer(device=0)
    sc.set_long_path(-1)
    nsm = torch.cuda.get_device_properties(0).multi_processor_count
    a = sc.score(codes, offs)
    n_auto = sc.stats().long_proteins
    assert 0 < n_auto <= nsm
    thr = np.sort(lens)[::-1][n_auto - 1]                   # shortest protein that went to the long path
    assert thr >= 1024 and (lens >= thr).sum() == n_auto
    d_codes, d_offs = torch.from_numpy(codes).cuda(), torch.from_numpy(offs).cuda()
    d_out = torch.zeros((len(lens), 160), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    sc.score_device(d_codes.data_ptr(), d_offs.data_ptr(), len(lens), int(offs[-1]), d_out.data_ptr())
    assert sc.stats().long_proteins == 2 * n_auto
    b = d_out.cpu().numpy().reshape(-1).view(plaac_b200.SUMMARY_DTYPE)
    sc.set_long_path(0)
    c = sc.score(codes, offs)
    assert sc.stats().long_proteins == 2 * n_auto
    sc.close()
    # long path (host API), long path (device API) and bucketed kernel: the same bytes -- the recurrences by the
    # binade-frame argument, the window columns because their sums are exact on the grid
    assert a.tobytes() == b.tobytes() == c.tobytes()
    # a large batch of short proteins: nothing is worth a CTA of its own
    codes, offs = synth.proteome(60000, seed=3, median=300.0, max_len=1700)  # chunks of 128 M residues: bound 1789
    big = np.concatenate([codes] * 12)
    boffs = np.concatenate([[0], np.cumsum(np.tile(np.diff(offs), 12))]).astype(np.int64)
    sc = plaac_b200.Scorer(device=0)
    sc.set_long_path(-1)
    sc.score(big, boffs)
    assert sc.stats().long_proteins == 0
    sc.close()


def test_long_path_with_exact_tie_constants():
    """Table constants that are exact round-half-even ties in the binades a long protein walks through (bits below
    the ulp exactly 1000...0): there a sum's rounding depends on its parity, the shift argument of the long-sequence
    path does not hold, and plaac_create must route those binades to the sequential redo (tie_binades).  The oracle
    does the same arithmetic sequentially.  (With the masks ignored, this test fails.)"""
    rng = np.random.default_rng(99)
    bg = synth.BG_SCER / synth.BG_SCER.sum()
    prd = synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for n in (9000, 20000):
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        for frac in (0.2, 0.6):
            st = int(n * frac)
            s[st:st + 180] = rng.choice(22, size=180, p=prd)
        seqs.append(s)
    codes, offs = plaac_b200.pack(seqs)
    P = plaac_b200.default_params()
    Q = orc.make_params()
    # binade [8192, 16384): ulp 2^-39, tie = an odd multiple of 2^-40; binade [16384, 32768): odd multiple of 2^-39
    ties = {10: -(2.0 + 3 * 2.0 ** -40),   # leucine, frequent: background and hmm0 emission, forward and Viterbi
            16: -(3.0 + 5 * 2.0 ** -39)}   # serine
    for code, v in ties.items():
        P.le[0][code] = v
        P.le0[code] = v
        Q.hmm1.le[0][code] = v
        Q.hmm0.le[0][code] = v
        Q.hmm0.le[1][code] = v
    P.llr[12] = 1.5 + 2.0 ** -40           # asparagine: the psum[] of the LLR search
    Q.llr[12] = P.llr[12]
    P.hydro2[1] = 0.25 + 2.0 ** -43        # alanine: the hydropathy sum (magnitudes 2^11..2^13 -> ulp 2^-41..2^-39)
    Q.hydro2[1] = P.hydro2[1]
    ref = orc.score_batch(Q, codes, offs)
    for min_len in (4096, 0):
        sc = plaac_b200.Scorer(P)
        sc.set_long_path(min_len)
        got = sc.score(codes, offs)
        st = sc.stats()
        sc.close()
        assert st.long_proteins == (2 if min_len else 0)
        _check(got, ref, f"tie constants, long_min={min_len}")


# Settings that once came from the environment and changed what a caller got back (a skipped role of the v3 kernel,
# ignored tie masks, another kernel or path): a variable left in a user's shell must not reach the results.
RETIRED_ENV = {"PLAAC_V3_MIX": "256", "PLAAC_SUMMARY_KERNEL": "2", "PLAAC_V3_OPT": "8", "PLAAC_V3_NT": "512",
               "PLAAC_LONG_TIES": "0", "PLAAC_NO_LONG_RES": "1"}


def test_retired_environment_variables_change_nothing(monkeypatch):
    """Records and per-residue arrays of a proteome with long proteins on the long-sequence path: a Scorer created with
    each retired variable set, and with all of them, gives the bytes of one created without them."""
    sc_, so = synth.proteome(2000, seed=31, median=300.0)
    lc, lo = synth.long_proteins(seed=1011, lengths=(1100, 2500, 9000))
    codes = np.concatenate([sc_, lc])
    offs = np.concatenate([so, lo[1:] + so[-1]])

    def run():
        sc = plaac_b200.Scorer()
        sc.set_long_path(1024)
        only = sc.score(codes, offs)
        summ, res = sc.score(codes, offs, per_residue=True)
        nlong = sc.stats().long_proteins
        sc.close()
        return only, summ, res, nlong

    want = run()
    assert want[3] == 2 * int((np.diff(offs) >= 1024).sum())
    for env in [{k: v} for k, v in RETIRED_ENV.items()] + [RETIRED_ENV]:
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        got = run()
        for k in env:
            monkeypatch.delenv(k)
        what = ", ".join(f"{k}={v}" for k, v in env.items())
        assert got[0].tobytes() == want[0].tobytes(), what
        assert got[1].tobytes() == want[1].tobytes(), what
        _residue_equal_bits(got[2], want[2], what)
        assert got[3] == want[3], what
