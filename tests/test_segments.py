"""Prion-like segments of the Viterbi parse (plaac_score_segments, Scorer.score_segments, the CLI's --segments).

A segment is a maximal run of 1s of the VIT column of per-residue mode, scored by the PRDscore rule (a sequential sum of
llr from 0.0).  The reference of every test here is that definition applied to a VIT column: the jar's own, the
oracle's, or the GPU's per-residue output."""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

import plaac_b200
from oracle import orc
from plaac_b200 import build as pb
from tests import jarvec, synth
from tests.test_host_cli import java_fmt

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


# ---------------------------------------------------------------------------------------------- the definition
def vit_runs(vit):
    """(start, end) arrays of the maximal runs of 1s of one VIT column (0-based, end inclusive)."""
    v = np.asarray(vit, dtype=np.int8)
    d = np.diff(np.r_[np.int8(0), v, np.int8(0)])
    return np.nonzero(d == 1)[0], np.nonzero(d == -1)[0] - 1


def run_score(llr, aa):
    """0.0 + llr[aa[0]] + ... in residue order (codes > 21 count as X)."""
    a = np.asarray(aa, dtype=np.int64)
    a = np.where(a > 21, 0, a)
    return float(np.add.accumulate(np.r_[0.0, np.asarray(llr, dtype=np.float64)[a]])[-1])


def reference_segments(codes, offsets, vit, llr):
    """The segments of a batch from its VIT column (residue index = index into codes)."""
    first, st, en, sc = [0], [], [], []
    for i in range(len(offsets) - 1):
        lo, hi = int(offsets[i]), int(offsets[i + 1])
        s, e = vit_runs(vit[lo - int(offsets[0]):hi - int(offsets[0])])
        for a, b in zip(s.tolist(), e.tolist()):
            st.append(a)
            en.append(b)
            sc.append(run_score(llr, codes[lo + a:lo + b + 1]))
        first.append(len(st))
    return {"first": np.array(first, np.int64), "start": np.array(st, np.int32), "end": np.array(en, np.int32),
            "score": np.array(sc, np.float64)}


def assert_same_segments(got, want, what):
    assert np.array_equal(got["first"], want["first"]), f"{what}: first differs"
    for k in ("start", "end"):
        assert np.array_equal(got[k], want[k]), f"{what}: {k} differs"
    g, w = np.asarray(got["score"], np.float64), np.asarray(want["score"], np.float64)
    bad = np.nonzero(g.view(np.uint64) != w.view(np.uint64))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(g)} scores differ, first {bad[:5].tolist()}"


def assert_prd_identity(rec, seg, what):
    """The segment holding the CORE is (prd_start, prd_end, prd_score) bit for bit; the longest is vit_maxrun long;
    a protein has no segment iff vit_maxrun is 0."""
    first = seg["first"]
    cnt = np.diff(first)
    lens = (seg["end"] - seg["start"] + 1).astype(np.int64)
    has = cnt > 0
    mx = np.zeros(len(rec), np.int64)
    mx[has] = np.maximum.reduceat(lens, first[:-1][has]) if has.any() else mx[has]
    assert np.array_equal(mx, rec["vit_maxrun"].astype(np.int64)), f"{what}: longest segment != vit_maxrun"
    assert np.array_equal(has, rec["vit_maxrun"] > 0), what
    core = np.nonzero(~np.isnan(rec["core_score"]))[0]
    pid = np.repeat(np.arange(len(rec)), cnt)
    hit = (seg["start"] == rec["prd_start"][pid]) & (seg["end"] == rec["prd_end"][pid])
    nprd = np.bincount(pid[hit], minlength=len(rec))
    assert np.all(nprd[core] == 1), f"{what}: a CORE without its PrD segment"
    assert np.all(nprd[np.isnan(rec["core_score"])] == 0), what
    k = np.nonzero(hit)[0]
    assert np.array_equal(seg["score"][k].view(np.uint64), rec["prd_score"][pid[k]].view(np.uint64)), f"{what}: PRDscore"


def llr_of(**kw):
    return np.array(orc.make_params(**kw).llr[:22], dtype=np.float64)


# ---------------------------------------------------------------------------------------------- CPU
def test_segments_struct_matches_the_header(tmp_path):
    src = tmp_path / "seg.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "plaac_cuda.h"\nint main(void){'
                   + "".join(f'printf("%zu\\n", offsetof(plaac_segments, {n}));' for n, _ in plaac_b200.Segments._fields_)
                   + 'printf("%zu\\n", sizeof(plaac_segments)); return 0;}\n')
    exe = tmp_path / "seg"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[:-1] == [getattr(plaac_b200.Segments, n).offset for n, _ in plaac_b200.Segments._fields_]
    assert got[-1] == C.sizeof(plaac_b200.Segments) == 48


def test_reference_runs_against_oracle_records():
    """The test's own reference against the oracle's records: the PrD segment is prd_* bit for bit, the longest run is
    vit_maxrun."""
    P = orc.make_params()
    for codes, offs in (synth.proteome(3000, seed=5), synth.repeat_proteome(300, seed=6), synth.edge_cases()):
        res = orc.residue_batch(P, codes, offs, nthreads=orc.max_threads())
        rec = orc.score_batch(P, codes, offs, nthreads=orc.max_threads())
        seg = reference_segments(codes, offs, res["vit"], llr_of())
        assert_prd_identity(rec, seg, "oracle")
    assert vit_runs([0, 1, 1, 0, 1]) [0].tolist() == [1, 4] and vit_runs([1, 1, 0, 1])[1].tolist() == [1, 3]
    assert run_score(llr_of(), [30, 0]) == 0.0 + llr_of()[0] + llr_of()[0]


@pytest.fixture(scope="module")
def cli():
    pb.build_lib()
    path = pb.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args):
    return subprocess.run([cli, *args], capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("extra, clash", [
    (["-p", "all"], "-p"), (["--variants", "v.txt"], "--variants"), (["--saturate"], "--saturate"),
    (["--gpu-ingest"], "--gpu-ingest"), (["--gpus", "2"], "--gpus > 1"),
])
def test_cli_rejects_segments_with(cli, tmp_path, extra, clash):
    """Rejected with status 2 before any device is opened (this runs without a GPU)."""
    fa = tmp_path / "a.fa"
    fa.write_text(">a\nMQQNNQQ\n")
    r = run(cli, "-i", str(fa), "--segments", str(tmp_path / "s.tsv"), *extra)
    assert r.returncode == 2, r.stderr
    assert f"--segments cannot be combined with {clash}" in r.stderr
    assert "CUDA" not in r.stderr and "device" not in r.stderr


# ---------------------------------------------------------------------------------------------- GPU
def records_bytes(a):
    return np.ascontiguousarray(a).view(np.uint8)


def check_batch(sc, codes, offs, want, what, rec_want=None, **kw):
    rec, seg = sc.score_segments(codes, offs, **kw)
    assert_same_segments(seg, want, what)
    if rec is not None:
        if rec_want is None:
            rec_want = sc.score(codes, offs)
        assert np.array_equal(records_bytes(rec), records_bytes(rec_want)), f"{what}: records differ from plaac_score's"
    return rec, seg


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prions_residue", "edge_residue", "edge_alt_residue", "long_residue"])
def test_segments_are_the_runs_of_the_jar_vit(which):
    enc, kw, prots = jarvec.scenario(which)
    codes, offs = plaac_b200.pack([c for _, c in enc])
    vit = np.concatenate([np.array(pr["vit"], np.uint8) for pr in prots])
    want = reference_segments(codes, offs, vit, llr_of(**kw))
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    for long_min in ((8192, 1024, 0, -1) if which == "long_residue" else (8192,)):
        sc.set_long_path(long_min)
        rec0 = sc.score(codes, offs)
        n0 = sc.stats().long_proteins
        check_batch(sc, codes, offs, want, f"{which}, long path {long_min}", rec_want=rec0, capacity=len(want["start"]))
        if which == "long_residue" and long_min == 1024:
            assert sc.stats().long_proteins - n0 == 2
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prions_summary", "edge_summary", "edge_alt_summary", "long_summary", "human_summary"])
def test_prd_segment_is_the_jar_prd(which):
    enc, kw, rows = jarvec.scenario(which)
    codes, offs = plaac_b200.pack([c for _, c in enc])
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    for long_min in ((4096, 0) if which == "long_summary" else (8192,)):
        sc.set_long_path(long_min)
        rec, seg = sc.score_segments(codes, offs)
        assert_prd_identity(rec, seg, which)
        n = 0
        for i, row in enumerate(rows):
            if int(row["PRDstart"]) <= 0:
                continue
            k = [j for j in range(seg["first"][i], seg["first"][i + 1])
                 if seg["start"][j] + 1 == int(row["PRDstart"]) and seg["end"][j] + 1 == int(row["PRDend"])]
            assert len(k) == 1, (which, row["SEQid"])
            assert seg["score"][k[0]] == jarvec.val(row["PRDscore"]), (which, row["SEQid"])
            n += 1
        assert n > 0 or which.startswith("edge")
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["proteome", "repeat", "edge"])
def test_segments_against_oracle_runs(which):
    codes, offs = {"proteome": lambda: synth.proteome(20000, seed=11), "repeat": lambda: synth.repeat_proteome(2000, seed=12),
                   "edge": synth.edge_cases}[which]()
    P = orc.make_params()
    res = orc.residue_batch(P, codes, offs, nthreads=orc.max_threads())
    want = reference_segments(codes, offs, res["vit"], llr_of())
    sc = plaac_b200.Scorer()
    rec, seg = check_batch(sc, codes, offs, want, which)
    if which == "proteome":
        assert len(seg["start"]) > 1000 and np.diff(seg["first"]).max() >= 2
    sc.close()


@pytest.mark.gpu
def test_every_path_gives_the_same_segments():
    """Long path at 1 024 and at the automatic threshold, kernel variant 1, independent -w / -W, a batch spread over many
    chunks, pinned outputs and no records."""
    codes, offs = synth.proteome(6000, seed=21)
    lc, lo = synth.long_proteins()
    codes = np.concatenate([codes, lc])
    offs = np.r_[offs, offs[-1] + lo[1:]]
    P = orc.make_params()
    res = orc.residue_batch(P, codes, offs, nthreads=orc.max_threads())
    want = reference_segments(codes, offs, res["vit"], llr_of())
    sc = plaac_b200.Scorer()
    rec0 = sc.score(codes, offs)
    for lm in (1024, -1, 0):
        sc.set_long_path(lm)
        n0 = sc.stats().long_proteins
        check_batch(sc, codes, offs, want, f"long path {lm}", rec_want=rec0)
        if lm == 1024:
            assert sc.stats().long_proteins - n0 > 2
    sc.set_long_path(8192)
    sc.set_chunk(1 << 20, 700)  # many chunks
    check_batch(sc, codes, offs, want, "small chunks", rec_want=rec0)
    rec, seg = sc.score_segments(codes, offs, summaries=False)
    assert rec is None
    assert_same_segments(seg, want, "no records")
    sc.set_chunk(256 << 20, 4 << 20)
    sc.set_kernel_variant(1)
    check_batch(sc, codes, offs, want, "kernel variant 1")  # (its records are its own: v1 is the reference-order anchor)
    sc.close()

    # pinned buffers everywhere (the raw call)
    sc = plaac_b200.Scorer()
    nprot, cnt = len(offs) - 1, len(want["start"])
    with plaac_b200.PinnedBuffer(len(codes)) as pc, plaac_b200.PinnedBuffer(nprot + 1, np.int64) as po, \
            plaac_b200.PinnedBuffer(nprot, plaac_b200.SUMMARY_DTYPE) as pr, plaac_b200.PinnedBuffer(nprot + 1, np.int64) as pf, \
            plaac_b200.PinnedBuffer(cnt, np.int32) as ps, plaac_b200.PinnedBuffer(cnt, np.int32) as pe, \
            plaac_b200.PinnedBuffer(cnt, np.float64) as pd:
        pc.array[:] = codes
        po.array[:] = offs
        g = plaac_b200.Segments(capacity=cnt, first=pf.ptr, start=ps.ptr, end=pe.ptr, score=pd.ptr, count=0)
        assert plaac_b200.lib().plaac_score_segments(sc._h, pc.ptr, po.ptr, nprot, pr.ptr, C.byref(g)) == 0
        assert g.count == cnt
        assert_same_segments({"first": pf.array.copy(), "start": ps.array.copy(), "end": pe.array.copy(), "score": pd.array.copy()},
                             want, "pinned")
        assert np.array_equal(records_bytes(pr.array), records_bytes(rec0))
    sc.close()

    # independent -w / -W (generic windows) and another core length
    kw = dict(ww1=31, ww2=51, core_len=40)
    P = orc.make_params(**kw)
    res = orc.residue_batch(P, codes, offs, nthreads=orc.max_threads())
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    check_batch(sc, codes, offs, reference_segments(codes, offs, res["vit"], llr_of(**kw)), "-w 31 -W 51 -c 40")
    sc.close()


def dense_batch(nprot=120, seed=31):
    """Proteins of alternating Q/N-rich and background blocks: dozens of segments per protein."""
    rng = np.random.default_rng(seed)
    bg, prd = synth.BG_SCER / synth.BG_SCER.sum(), synth.PRD_28 / synth.PRD_28.sum()
    seqs = []
    for _ in range(nprot):
        parts = []
        for _ in range(int(rng.integers(20, 60))):
            parts.append(rng.choice(22, size=int(rng.integers(25, 90)), p=prd))
            parts.append(rng.choice(22, size=int(rng.integers(30, 120)), p=bg))
        seqs.append(np.concatenate(parts).astype(np.uint8))
    return plaac_b200.pack(seqs)


@pytest.mark.gpu
def test_overflowing_the_slot_entries_gives_the_roomy_result():
    codes, offs = dense_batch()
    P = orc.make_params()
    res = orc.residue_batch(P, codes, offs, nthreads=orc.max_threads())
    want = reference_segments(codes, offs, res["vit"], llr_of())
    # one chunk keeps nres / 2048 + 1024 entries: far fewer than the batch's segments
    assert len(want["start"]) > 2 * (int(offs[-1]) // 2048 + 1024)
    sc = plaac_b200.Scorer()
    rec0 = sc.score(codes, offs)
    check_batch(sc, codes, offs, want, "overflowing", rec_want=rec0)
    for lm in (1024, -1):
        sc.set_long_path(lm)
        check_batch(sc, codes, offs, want, f"overflowing, long path {lm}", rec_want=rec0)
    sc.set_long_path(8192)
    sc.set_chunk(1 << 20, 6)  # roomy: a few proteins per chunk
    check_batch(sc, codes, offs, want, "roomy", rec_want=rec0)
    sc.close()


@pytest.mark.gpu
def test_capacity_and_argument_errors():
    codes, offs = synth.proteome(3000, seed=41)
    sc = plaac_b200.Scorer()
    _, full = sc.score_segments(codes, offs, capacity=10 ** 6)
    count = len(full["start"])
    assert count > 50
    L, nprot = plaac_b200.lib(), len(offs) - 1

    def raw(cap, codes=codes, offs=offs, nprot=nprot, first=True, arrays=True):
        f = np.full(nprot + 1, -7, np.int64)
        s, e, d = np.full(max(cap, 1), -7, np.int32), np.full(max(cap, 1), -7, np.int32), np.full(max(cap, 1), -7.0)
        g = plaac_b200.Segments(capacity=cap, first=f.ctypes.data if first else None, start=s.ctypes.data if arrays else None,
                                end=e.ctypes.data if arrays else None, score=d.ctypes.data if arrays else None, count=-1)
        rc = L.plaac_score_segments(sc._h, codes.ctypes.data, offs.ctypes.data, nprot, None, C.byref(g))
        return rc, g.count, {"first": f, "start": s, "end": e, "score": d}

    for cap in (0, 1, count // 2, count - 1, count):
        rc, n, got = raw(cap)
        assert rc == 0 and n == count, cap
        assert np.array_equal(got["first"], full["first"]), cap
        for k in ("start", "end", "score"):
            assert np.array_equal(got[k][:cap], full[k][:cap]), (cap, k)
        assert np.all(got["start"][cap:] == -7)
    rc, n, got = raw(5, nprot=0)
    assert rc == 0 and n == 0 and got["first"][0] == 0
    rc, n, got = raw(0, nprot=0, first=False, arrays=False)
    assert rc == 0 and n == 0
    assert raw(-1)[0] == -1
    assert raw(5, first=False)[0] == -1
    assert raw(5, arrays=False)[0] == -1
    assert raw(0, arrays=False)[0] == 0
    # Python: a too small capacity is retried with room for all
    _, again = sc.score_segments(codes, offs, capacity=3)
    assert_same_segments(again, full, "retried")
    # bytes > 21 are X: everything written, then PLAAC_E_INVALID
    bad = codes.copy()
    bad[offs[7] + 3] = 40
    bad[offs[100] + 1] = 200
    fixed = np.where(bad > 21, 0, bad).astype(np.uint8)
    _, want = sc.score_segments(fixed, offs)
    rec_fixed = sc.score(fixed, offs)
    rec = np.zeros(nprot, plaac_b200.SUMMARY_DTYPE)
    cnt = len(want["start"])
    f, s, e, d = np.zeros(nprot + 1, np.int64), np.zeros(cnt, np.int32), np.zeros(cnt, np.int32), np.zeros(cnt)
    g = plaac_b200.Segments(capacity=cnt, first=f.ctypes.data, start=s.ctypes.data, end=e.ctypes.data, score=d.ctypes.data)
    assert L.plaac_score_segments(sc._h, bad.ctypes.data, offs.ctypes.data, nprot, rec.ctypes.data, C.byref(g)) == -1
    assert g.count == cnt
    assert_same_segments({"first": f, "start": s, "end": e, "score": d}, want, "bytes > 21")
    assert np.array_equal(records_bytes(rec), records_bytes(rec_fixed))
    sc.close()


def bench_batch(nprot):
    import torch

    import bench

    codes, offsets, ntotal = bench.synth_shard(plaac_b200.lib(), torch.device("cuda", 0), 0, nprot)
    torch.cuda.synchronize()
    return codes[:ntotal].cpu().numpy(), offsets.cpu().numpy()


@pytest.mark.gpu
def test_bench_distribution_against_the_gpu_per_residue_vit():
    codes, offs = bench_batch(200_000)
    sc = plaac_b200.Scorer()
    rec, res = sc.score(codes, offs, per_residue=True)
    want = reference_segments(codes, offs, res["vit"], llr_of())
    check_batch(sc, codes, offs, want, "200 k bench proteins", rec_want=rec)
    sc.close()


@pytest.mark.gpu
def test_bench_shard_prd_identity():
    """The benchmark's own shard (12.5 M proteins, 4.39 G residues): per protein the longest segment is vit_maxrun long,
    there is none iff vit_maxrun is 0, and the segment holding the CORE is the PrD."""
    codes, offs = bench_batch(12_500_000)
    sc = plaac_b200.Scorer()
    rec, seg = sc.score_segments(codes, offs)
    assert offs[-1] > 2**32 and len(seg["start"]) > 0
    assert_prd_identity(rec, seg, "bench shard")
    ref = sc.score(codes[:int(offs[200_000])], offs[:200_001])
    assert np.array_equal(records_bytes(rec[:200_000]), records_bytes(ref))
    sc.close()


def classic_fasta(tmp_path):
    with open(os.path.join(GOLD, "classic_prions.json")) as f:
        golden = json.load(f)
    fa = tmp_path / "classic.fa"
    fa.write_text("".join(f">{p['name']}\n{p['seq']}\n" for p in golden["proteins"]))
    return fa


@pytest.mark.gpu
@pytest.mark.parametrize("rank", [False, True])
def test_cli_segments_file_is_the_table_of_the_vit_column(cli, tmp_path, rank):
    fa = classic_fasta(tmp_path)
    extra = ["--rank"] if rank else []
    plain = run(cli, "-i", str(fa), *extra)
    seg_path = tmp_path / "seg.tsv"
    withseg = run(cli, "-i", str(fa), "--segments", str(seg_path), *extra)
    assert plain.returncode == 0 and withseg.returncode == 0, withseg.stderr
    assert withseg.stdout == plain.stdout
    # the same table from -p all: VIT runs, llr sums of the residues, PrD of the summary rows
    per = run(cli, "-i", str(fa), "-p", "all")
    assert per.returncode == 0
    lines = [ln.split("\t") for ln in per.stdout.splitlines() if ln and not ln.startswith("#")]
    head = lines[0]
    iv, ia, isq = head.index("VIT"), head.index("AA"), head.index("SEQid")
    cols = {}
    for ln in lines[1:]:
        cols.setdefault(ln[isq], ([], []))
        cols[ln[isq]][0].append(int(ln[iv]))
        cols[ln[isq]][1].append(ln[ia])
    summ = [ln.split("\t") for ln in plain.stdout.splitlines() if ln and not ln.startswith("#")]
    sh = summ[0]
    prd = {r[sh.index("SEQid")]: (int(r[sh.index("PRDstart")]), int(r[sh.index("PRDend")])) for r in summ[1:]}
    llr = llr_of()  # (alpha = 1: the input's composition does not enter the tables)
    want = ["SEQid\tSEGstart\tSEGend\tSEGlen\tSEGscore\tPRD"]
    for name, (vit, aa) in cols.items():
        codes = orc.encode("".join(aa))
        for a, b in zip(*vit_runs(vit)):
            want.append(f"{name}\t{a + 1}\t{b + 1}\t{b - a + 1}\t{java_fmt(run_score(llr, codes[a:b + 1]), 3)}\t"
                        f"{1 if prd[name] == (a + 1, b + 1) else 0}")
    got = seg_path.read_text().splitlines()
    assert got == want
    mot3 = [ln for ln in got if ln.startswith("Mot3p\t")]
    assert [ln.split("\t")[1:3] for ln in mot3] == [["1", "296"], ["413", "442"]]
