"""Sequence variants (plaac_score_variants, Scorer.score_variants, saturation(), the CLI's --variants / --saturate).

Record v of a variant call is, byte for byte, the record plaac_score gives for the mutated protein, so the oracle of
every GPU test here is the existing path on a batch materialised with numpy."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plaac_b200
from oracle import orc
from plaac_b200 import build as pb
from tests import parity, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NT = max(1, min(32, os.cpu_count() or 1))
AA = "XACDEFGHIKLMNPQRSTVWY*"
P_, A_, Q_, N_, X_, STOP = 13, 1, 14, 12, 0, 21
CHARGED = [3, 4, 9, 15]  # D E K R


# ---------------------------------------------------------------------------------------------- helpers
def materialise(codes, offsets, protein, first_sub, pos, code):
    """The mutated proteins as one ordinary batch."""
    seqs = []
    for v in range(len(protein)):
        p = int(protein[v])
        s = codes[offsets[p]:offsets[p + 1]].copy()
        a, b = int(first_sub[v]), int(first_sub[v + 1])
        s[pos[a:b]] = code[a:b]
        seqs.append(s)
    return plaac_b200.pack(seqs)


def as_rows(a):
    return np.ascontiguousarray(a).view(np.uint8).reshape(len(a), -1)


def assert_same_bytes(got, want, what):
    g, w = as_rows(got), as_rows(want)
    assert g.shape == w.shape, what
    bad = np.nonzero((g != w).any(axis=1))[0]
    assert len(bad) == 0, f"{what}: {len(bad)} of {len(g)} records differ, first {bad[:10].tolist()}"


def build_variants(codes, offsets, wt, nvar, seed):
    """~nvar variants in random protein order covering the kinds the contract names."""
    rng = np.random.default_rng(seed)
    nprot = len(offsets) - 1
    lens = np.diff(offsets)
    specs = []  # (protein, [(pos, code), ...])
    pick = lambda: int(rng.integers(0, nprot))  # noqa: E731
    kinds = 0
    while len(specs) < nvar:
        p = pick()
        n = int(lens[p])
        s = codes[offsets[p]:offsets[p + 1]]
        k = kinds % 12
        kinds += 1
        if n == 0:
            continue
        if k == 0:
            specs.append((p, []))
        elif k == 1:
            specs.append((p, [(int(rng.integers(0, n)), int(rng.integers(0, 22)))]))
        elif k == 2 and n >= 2:
            a, b = sorted(rng.choice(n, 2, replace=False).tolist())
            specs.append((p, [(a, int(rng.integers(1, 21))), (b, int(rng.integers(0, 22)))]))
        elif k == 3:
            specs.append((p, [(0, int(rng.integers(0, 22)))]))
            specs.append((p, [(n - 1, int(rng.integers(0, 22)))]))
        elif k == 4:
            # create / destroy PP and PxP (the PAPA proline flags of the neighbours)
            prol = np.nonzero(s == P_)[0]
            if len(prol):
                i = int(rng.choice(prol))
                for j in (i - 2, i - 1, i + 1, i + 2):
                    if 0 <= j < n:
                        specs.append((p, [(j, P_)]))
                specs.append((p, [(i, A_)]))
        elif k == 5:
            i = int(rng.integers(0, n))
            specs.append((p, [(i, int(rng.choice(CHARGED)))]))
            ch = np.nonzero(np.isin(s, CHARGED))[0]
            if len(ch):
                specs.append((p, [(int(rng.choice(ch)), int(rng.choice([A_, Q_, N_, X_]))) ]))
        elif k == 6:
            i = int(rng.integers(0, n))
            specs.append((p, [(i, int(rng.choice([Q_, N_])))]))
            qn = np.nonzero((s == Q_) | (s == N_))[0]
            if len(qn):
                specs.append((p, [(int(rng.choice(qn)), int(rng.integers(1, 21)))]))
        elif k == 7:
            i = int(rng.integers(0, n))
            specs.append((p, [(i, X_)]))
            specs.append((p, [(i, STOP)]))
            xs = np.nonzero((s == X_) | (s == STOP))[0]
            if len(xs):
                specs.append((p, [(int(rng.choice(xs)), int(rng.integers(1, 21)))]))
        elif k == 8:
            # inside and outside the wild type's CORE
            cs, ce = int(wt["core_start"][p]), int(wt["core_end"][p])
            if cs >= 0:
                specs.append((p, [(int(rng.integers(cs, ce + 1)), int(rng.choice([A_, P_, Q_, CHARGED[0]])))]))
                out = [i for i in (cs - 1, ce + 1, 0, n - 1) if 0 <= i < n and not cs <= i <= ce]
                if out:
                    specs.append((p, [(out[int(rng.integers(0, len(out)))], int(rng.integers(1, 21)))]))
        elif k == 9:
            m = int(min(n, rng.integers(3, 60)))
            at = np.sort(rng.choice(n, m, replace=False))
            specs.append((p, [(int(i), int(rng.integers(0, 22))) for i in at]))
        elif k == 10 and specs:
            specs.append(specs[int(rng.integers(0, len(specs)))])  # a repeated identical variant
        elif k == 11:
            specs.append((p, [(int(rng.integers(0, n)), int(s[int(rng.integers(0, n))]))]))  # often a silent change
    order = rng.permutation(len(specs))
    specs = [specs[i] for i in order]
    protein = np.array([p for p, _ in specs], dtype=np.int32)
    first_sub = np.zeros(len(specs) + 1, dtype=np.int64)
    np.cumsum([len(sub) for _, sub in specs], out=first_sub[1:])
    pos = np.array([q for _, sub in specs for q, _ in sub], dtype=np.int32)
    code = np.array([c for _, sub in specs for _, c in sub], dtype=np.uint8)
    return protein, first_sub, pos, code


def reference_batch():
    """Edge-case lengths 1..257 around every window size, typical lengths, and proteins of 9 k, 20 k and 40 k residues."""
    parts = [synth.edge_cases(), synth.proteome(300, seed=41), synth.long_proteins(seed=43, lengths=(9000, 20000, 40000))]
    seqs = []
    for c, o in parts:
        seqs += [c[o[i]:o[i + 1]] for i in range(len(o) - 1)]
    return plaac_b200.pack(seqs)


@pytest.fixture(scope="module")
def scorer():
    s = plaac_b200.Scorer()
    yield s
    s.close()


@pytest.fixture(scope="module")
def case(scorer):
    codes, offs = reference_batch()
    wt = scorer.score(codes, offs)
    var = build_variants(codes, offs, wt, 3000, seed=5)
    mc, mo = materialise(codes, offs, *var)
    return codes, offs, var, mc, mo


# ---------------------------------------------------------------------------------------------- CPU
def test_variants_struct_matches_header(tmp_path):
    assert C.sizeof(plaac_b200.Variants) == 40
    src = tmp_path / "layout.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "plaac_cuda.h"\nint main(void){printf("%zu %zu %zu %zu %zu %zu\\n",'
                   'sizeof(plaac_variants), offsetof(plaac_variants, nvar), offsetof(plaac_variants, protein),'
                   'offsetof(plaac_variants, first_sub), offsetof(plaac_variants, pos), offsetof(plaac_variants, code));return 0;}\n')
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    V = plaac_b200.Variants
    assert got == [C.sizeof(V)] + [getattr(V, n).offset for n, _ in V._fields_] == [40, 0, 8, 16, 24, 32]


def test_saturation_counts_and_order():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MAX*Q", strip_stop=False), plaac_b200.encode(""),
                                   plaac_b200.encode("QN")])
    protein, first_sub, pos, code = plaac_b200.saturation(codes, offs)
    # protein 0: WT + 19 (M) + 19 (A) + 20 (X) + 20 (*) + 19 (Q); protein 1: WT only; protein 2: WT + 19 + 19
    assert len(protein) == 98 + 1 + 39
    assert protein.tolist() == [0] * 98 + [1] + [2] * 39
    nsub = np.diff(first_sub)
    assert nsub[0] == 0 and nsub[98] == 0 and nsub[99] == 0 and (nsub[1:98] == 1).all() and (nsub[100:] == 1).all()
    assert first_sub[0] == 0 and first_sub[-1] == len(pos) == len(code) == 97 + 38
    assert pos[:19].tolist() == [0] * 19 and code[:19].tolist() == [c for c in range(1, 21) if c != 11]
    assert pos[38:58].tolist() == [2] * 20 and code[38:58].tolist() == list(range(1, 21))  # X: all 20
    assert pos[58:78].tolist() == [3] * 20 and code[58:78].tolist() == list(range(1, 21))  # '*': all 20
    assert (np.diff(pos[:97]) >= 0).all()
    # a subset, in the order given
    pr, fs, ps, cs = plaac_b200.saturation(codes, offs, proteins=[2, 0])
    assert pr.tolist() == [2] * 39 + [0] * 98
    assert len(ps) == 38 + 97 and fs[-1] == len(ps)


@pytest.fixture(scope="module")
def cli():
    pb.build_lib()
    path = pb.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args):
    return subprocess.run([cli, *args], capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("line, why", [("a\tM1A,Q2", "line 2"), ("a\tQ2Z", "unknown residue letter"), ("a M1A", "SEQid<TAB>spec"),
                                       ("a\tM0A", "1-based position"), ("a\tMxA", "1-based position"),
                                       ("a\tM1A,M1C", "substituted twice")])
def test_cli_variant_file_syntax_errors(cli, tmp_path, line, why):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    vf = tmp_path / "v.txt"
    vf.write_text("a\tWT\n" + line + "\n")
    r = run(cli, "-s", "-i", str(fa), "--variants", str(vf))
    assert r.returncode == 2
    assert "line 2" in r.stderr and why in r.stderr, r.stderr
    assert "SEQid" not in r.stdout


@pytest.mark.parametrize("extra", [["-p", "all"], ["--rank"], ["--rank-core"], ["--gpu-ingest"], ["--gpus", "2"]])
@pytest.mark.parametrize("mode", ["--saturate", "--variants"])
def test_cli_rejected_combinations(cli, tmp_path, extra, mode):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    vf = tmp_path / "v.txt"
    vf.write_text("a\tWT\n")
    args = [mode] + ([str(vf)] if mode == "--variants" else [])
    r = run(cli, "-s", "-i", str(fa), *args, *extra)
    assert r.returncode == 2 and "cannot be combined" in r.stderr, r.stderr
    assert r.stdout == ""


def test_cli_variants_with_saturate_rejected(cli, tmp_path):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    vf = tmp_path / "v.txt"
    vf.write_text("a\tWT\n")
    r = run(cli, "-s", "-i", str(fa), "--saturate", "--variants", str(vf))
    assert r.returncode == 2 and "cannot be combined" in r.stderr


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_records_equal_the_materialised_batch(scorer, case):
    codes, offs, var, mc, mo = case
    want = scorer.score(mc, mo)
    assert (want["core_start"] >= 0).sum() > 20  # the batch has proteins with a CORE
    got = scorer.score_variants(codes, offs, *var)
    assert_same_bytes(got, want, "variants")
    # variant slices spread over many chunks
    sc = plaac_b200.Scorer()
    try:
        sc.set_chunk(0, 400)
        got = sc.score_variants(codes, offs, *var)
    finally:
        sc.close()
    assert len(var[0]) >= 5 * 400
    assert_same_bytes(got, want, "variants, 400 per chunk")


@pytest.mark.gpu
def test_long_path_setting_of_the_materialising_ctx(case):
    """Long variants go through the cluster kernels when materialised (threshold 1024 / default) and through whatever the
    automatic rule picks in the variant call: same bytes.  The call leaves the ctx's own setting as it was."""
    codes, offs, var, mc, mo = case
    assert (np.diff(mo) >= 9000).sum() > 5
    ref = plaac_b200.Scorer()
    vs = plaac_b200.Scorer()
    try:
        got = vs.score_variants(codes, offs, *var)
        for thr in (1024, None):
            if thr is not None:
                ref.set_long_path(thr)
            before = ref.stats().long_proteins
            want = ref.score(mc, mo)
            assert ref.stats().long_proteins > before
            assert_same_bytes(got, want, f"long path {thr}")
        vs.set_long_path(1024)
        vs.score_variants(codes, offs, *var)
        before = vs.stats().long_proteins
        vs.score(mc, mo)
        assert vs.stats().long_proteins - before == (np.diff(mo) >= 1024).sum()
    finally:
        ref.close()
        vs.close()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["pinned", "generic_windows", "kernel_variant_1"])
def test_other_code_paths(case, how):
    codes, offs, var, mc, mo = case
    params = plaac_b200.default_params(ww1=31, ww2=51) if how == "generic_windows" else None
    sc = plaac_b200.Scorer(params)
    try:
        if how == "kernel_variant_1":
            sc.set_kernel_variant(1)
        want = sc.score(mc, mo)
        if how == "pinned":
            n = len(var[0])
            with plaac_b200.PinnedBuffer(n, dtype=plaac_b200.SUMMARY_DTYPE) as buf:
                got = sc.score_variants(codes, offs, *var, out=buf.array).copy()
        else:
            got = sc.score_variants(codes, offs, *var)
    finally:
        sc.close()
    assert_same_bytes(got, want, how)


@pytest.mark.gpu
def test_saturation_of_the_classic_prions_against_the_oracle(scorer, golden):
    seqs = [plaac_b200.encode(p["seq"]) for p in golden["proteins"]]
    codes, offs = plaac_b200.pack(seqs)
    var = plaac_b200.saturation(codes, offs)
    assert len(var[0]) > 30000
    got = scorer.score_variants(codes, offs, *var)
    mc, mo = materialise(codes, offs, *var)
    P = orc.make_params()
    ref = orc.score_batch(P, mc, mo, nthreads=NT)
    bad, nties = parity.compare_with_tie_classes(P, mc, mo, got.copy(), ref, orc.INT_FIELDS, orc.DBL_FIELDS)
    assert not bad, "\n".join(bad[:20])
    assert nties <= len(got) // 100


def _call(sc, codes, offs, nprot, protein, first_sub, pos, code, nvar, out):
    V = plaac_b200.Variants(nvar=nvar, protein=protein, first_sub=first_sub, pos=pos, code=code)
    rc = plaac_b200.lib().plaac_score_variants(sc._h, codes, offs, nprot, C.byref(V), out)
    return rc, plaac_b200.lib().plaac_last_error(sc._h).decode()


@pytest.mark.gpu
def test_invalid_inputs(scorer):
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDQQNKLLAPQ"), plaac_b200.encode("ACDEFG")])
    out = np.zeros(8, dtype=plaac_b200.SUMMARY_DTYPE)
    arr = lambda a, t: np.ascontiguousarray(a, dtype=t)  # noqa: E731

    def call(protein, first_sub, pos, code, nvar=None, null=()):
        a = [arr(protein, np.int32), arr(first_sub, np.int64), arr(pos, np.int32), arr(code, np.uint8)]
        ptrs = [None if i in null else x.ctypes.data for i, x in enumerate(a)]
        return _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, *ptrs, len(a[0]) if nvar is None else nvar, out.ctypes.data)

    ok = ([0, 1], [0, 1, 2], [3, 5], [1, 2])
    assert call(*ok)[0] == 0
    cases = {
        "protein index": ([0, 2], [0, 1, 2], [3, 5], [1, 2]),
        "negative protein index": ([-1, 1], [0, 1, 2], [3, 5], [1, 2]),
        "position outside": ([0, 1], [0, 1, 2], [3, 6], [1, 2]),
        "negative position": ([0, 1], [0, 1, 2], [-1, 5], [1, 2]),
        "not increasing": ([0, 1], [0, 2, 2], [3, 3], [1, 2]),
        "decreasing": ([0, 1], [0, 2, 2], [5, 3], [1, 2]),
        "code > 21": ([0, 1], [0, 1, 2], [3, 5], [1, 22]),
        "first_sub[0] != 0": ([0, 1], [1, 1, 2], [3, 5], [1, 2]),
        "first_sub decreases": ([0, 1], [0, 2, 1], [3, 5], [1, 2]),
    }
    want_index = {"protein index": 1, "negative protein index": 0, "position outside": 1, "negative position": 0,
                  "not increasing": 0, "decreasing": 0, "code > 21": 1, "first_sub[0] != 0": 0, "first_sub decreases": 1}
    for what, a in cases.items():
        rc, msg = call(*a)
        assert rc == -1, what
        assert f"variant {want_index[what]}" in msg, (what, msg)
    for k in range(4):
        rc, msg = call(*ok, null=(k,))
        assert rc == -1 and "NULL" in msg, k
    rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, None, None, None, None, 0, None)
    assert rc == 0
    with pytest.raises(plaac_b200.PlaacError, match="variant 0: position 99"):
        scorer.score_variants(codes, offs, [0], [0, 1], [99], [1])


@pytest.mark.gpu
def test_invalid_reference_bytes_as_plaac_score(scorer):
    codes, offs = reference_batch()
    codes = codes.copy()
    codes[offs[3] + 1] = 30
    codes[offs[50] + 7] = 200
    var = build_variants(codes, offs, scorer_wt(scorer, codes, offs), 600, seed=9)
    mc, mo = materialise(codes, offs, *var)
    want = np.zeros(len(var[0]), dtype=plaac_b200.SUMMARY_DTYPE)
    rc_ref = plaac_b200.lib().plaac_score(scorer._h, mc.ctypes.data, mo.ctypes.data, len(mo) - 1, want.ctypes.data, None)
    got = np.zeros(len(var[0]), dtype=plaac_b200.SUMMARY_DTYPE)
    a = [np.ascontiguousarray(x) for x in var]
    rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, len(offs) - 1, *[x.ctypes.data for x in a], len(a[0]), got.ctypes.data)
    assert rc_ref == -1 and rc == -1 and "> 21" in msg
    assert_same_bytes(got, want, "invalid reference bytes")


def scorer_wt(scorer, codes, offs):
    wt = np.zeros(len(offs) - 1, dtype=plaac_b200.SUMMARY_DTYPE)
    plaac_b200.lib().plaac_score(scorer._h, codes.ctypes.data, offs.ctypes.data, len(offs) - 1, wt.ctypes.data, None)
    return wt


# ---------------------------------------------------------------------------------------------- CLI on the GPU
def _fasta(names, seqs):
    return "".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in zip(names, seqs))


def _small_fasta(golden):
    rng = np.random.default_rng(17)
    names = [p["name"] for p in golden["proteins"][:2]] + ["rand1", "rand2"]
    seqs = [p["seq"].rstrip("*") for p in golden["proteins"][:2]]
    seqs += ["".join(AA[c] for c in rng.integers(1, 21, n)) for n in (70, 130)]
    seqs[3] = seqs[3][:40] + "X" + seqs[3][41:]
    return names, seqs


@pytest.mark.gpu
def test_cli_saturate_and_variants_match_the_materialised_fasta(cli, tmp_path, golden):
    names, seqs = _small_fasta(golden)
    fa = tmp_path / "small.fa"
    fa.write_text(_fasta(names, seqs))
    bg = tmp_path / "bg.txt"
    bg.write_text("".join(f"{v}\n" for v in synth.BG_HUMAN_COUNTS))
    # --saturate: every record, the order of saturation()
    sat_names, sat_seqs = [], []
    for n, s in zip(names, seqs):
        sat_names.append(f"{n}:WT")
        sat_seqs.append(s)
        for i, r in enumerate(s):
            for c in AA[1:21]:
                if c != r:
                    sat_names.append(f"{n}:{r}{i + 1}{c}")
                    sat_seqs.append(s[:i] + c + s[i + 1:])
    mat = tmp_path / "sat.fa"
    mat.write_text(_fasta(sat_names, sat_seqs))
    # --variants: a mixed file, lines of one record apart, lower case, unsorted tokens
    s0, s2 = seqs[0], seqs[2]
    lines = [(names[2], f"{s2[0]}1P"), (names[0], "WT"), (names[2], f"{s2[5].lower()}6q,{s2[1]}2n"), (names[0], f"{s0[9]}10X"),
             (names[2], "wt"), (names[0], f"{s0[0]}1A,{s0[-1]}{len(s0)}X"), (names[0], f"{s0[19]}20*"), (names[0], "WT")]
    # (no '*' at the last position: the materialised FASTA's reader would strip it as a stop codon)
    vf = tmp_path / "v.txt"
    vf.write_text("".join(f"{n}\t{sp}\n" for n, sp in lines))
    var_names, var_seqs = [], []
    for rec in (0, 2):  # record order, then file order
        for n, sp in lines:
            if n != names[rec]:
                continue
            s = list(seqs[rec])
            if sp.upper() != "WT":
                for tok in sp.upper().split(","):
                    s[int(tok[1:-1]) - 1] = tok[-1]
            var_names.append(f"{n}:{sp.upper()}")
            var_seqs.append("".join(s))
    vmat = tmp_path / "vmat.fa"
    vmat.write_text(_fasta(var_names, var_seqs))
    for extra in (["-a", "1"], ["-B", str(bg)], ["-B", str(bg), "-a", "0.5"]):
        for mode, m in ((["--saturate"], mat), (["--variants", str(vf)], vmat)):
            a = run(cli, "-s", "-i", str(fa), *mode, *extra)
            b = run(cli, "-s", "-i", str(m), *extra)
            assert a.returncode == 0 and b.returncode == 0, a.stderr + b.stderr
            al, bl = a.stdout.split("\n"), b.stdout.split("\n")
            assert len(al) == len(bl) > 10 if mode[0] == "--saturate" else len(al) == len(bl) == len(var_names) + 2
            assert al == bl, (mode, extra, next((x, y) for x, y in zip(al, bl) if x != y))
    # several batches: the same table
    a = run(cli, "-s", "-i", str(fa), "--saturate", "--batch-mb", "1")
    b = run(cli, "-s", "-i", str(mat))
    assert a.stdout == b.stdout


@pytest.mark.gpu
def test_cli_errors_that_need_a_record(cli, tmp_path, golden):
    names, seqs = _small_fasta(golden)
    fa = tmp_path / "small.fa"
    fa.write_text(_fasta(names, seqs))
    wrong = "A" if seqs[1][4] != "A" else "C"
    for lines, why in (([f"{names[1]}\tWT", f"{names[1]}\t{wrong}5C"], "line 2"),
                       ([f"{names[0]}\tWT", f"{names[1]}\t{seqs[1][0]}{len(seqs[1]) + 1}A"], "line 2"),
                       ([f"{names[0]}\tWT", "nosuchprotein\tWT"], "line 2")):
        vf = tmp_path / "v.txt"
        vf.write_text("\n".join(lines) + "\n")
        r = run(cli, "-s", "-i", str(fa), "--variants", str(vf))
        assert r.returncode == 2 and why in r.stderr, r.stderr
        assert [l for l in r.stdout.split("\n") if l and not l.startswith("SEQid")] == [], r.stdout
