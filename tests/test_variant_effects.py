"""Variant effects (plaac_score_variant_effects, Scorer.variant_effects, saturation_map(), the CLI's --effects).

An effect is a variant's record minus its wild type's, so the oracle of every GPU test here is the existing variant call
and plaac_score on the reference, subtracted in numpy."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plaac_b200
from plaac_b200 import build as pb
from tests.test_host_cli import java_fmt
from tests.test_variants import build_variants, reference_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AA = "XACDEFGHIKLMNPQRSTVWY*"
DOUBLES = [n for n in plaac_b200.SUMMARY_DTYPE.names if plaac_b200.SUMMARY_DTYPE[n] == np.float64]
ALL = (1 << 14) - 1
CLI_NAMES = ["LLR", "COREscore", "PRDscore", "HMMall", "HMMvit", "FImeanhydro", "FImeancharge", "FImeancombo",
             "PAPAcombo", "PAPAprop", "PAPAfi", "PAPAllr", "PAPAllr2", "COREchange"]


def expected(var_rec, wild_rec, protein, names):
    """The effects the contract defines, computed in numpy from records."""
    w = wild_rec[np.asarray(protein, dtype=np.int64)]
    out = np.zeros(len(var_rec), dtype=plaac_b200.effects_dtype(sum(1 << plaac_b200.EFFECT_COLUMNS.index(n) for n in names)))
    for n in out.dtype.names:
        if n == "core_change":
            out[n] = (~np.isnan(var_rec["core_score"])).astype(np.float64) - (~np.isnan(w["core_score"])).astype(np.float64)
        else:
            with np.errstate(invalid="ignore"):
                out[n] = var_rec[n] - w[n]
    return out


def assert_same_effects(got, want, what):
    """Bitwise, with every NaN equal to every other NaN."""
    assert got.dtype.names == want.dtype.names, what
    for n in want.dtype.names:
        g, w = np.ascontiguousarray(got[n]), np.ascontiguousarray(want[n])
        gn, wn = np.isnan(g), np.isnan(w)
        bad = np.nonzero((gn != wn) | (~gn & (g.view(np.uint64) != w.view(np.uint64))))[0]
        assert len(bad) == 0, f"{what}, {n}: {len(bad)} of {len(g)} differ, first {bad[:10].tolist()}"


# ---------------------------------------------------------------------------------------------- CPU
def test_effect_bits_follow_the_record_and_the_header(tmp_path):
    assert list(plaac_b200.EFFECT_COLUMNS) == DOUBLES + ["core_change"] and len(DOUBLES) == 13
    macros = ["LLR", "CORE_SCORE", "PRD_SCORE", "HMM_ALL", "HMM_VIT", "FI_MEANHYDRO", "FI_MEANCHARGE", "FI_MEANCOMBO",
              "PAPA_COMBO", "PAPA_PROP", "PAPA_FI", "PAPA_LLR", "PAPA_LLR2", "CORE_CHANGE"]
    src = tmp_path / "bits.c"
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "plaac_cuda.h"\nint main(void){'
                   + "".join(f'printf("%d\\n", PLAAC_EFFECT_{m});' for m in macros)
                   + "".join(f'printf("%zu\\n", offsetof(plaac_summary, {n}));' for n in DOUBLES) + "return 0;}\n")
    exe = tmp_path / "bits"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[:14] == [1 << k for k in range(14)]
    # bits 0..12 are the doubles in declaration order, as SUMMARY_DTYPE lists its f8 fields
    offs = got[14:]
    assert offs == sorted(offs) and np.all(np.diff(offs) == 8)
    assert offs == [plaac_b200.SUMMARY_DTYPE.fields[n][1] for n in DOUBLES]
    dt = plaac_b200.effects_dtype((1 << 13) | (1 << 1) | 1)
    assert dt.names == ("llr", "core_score", "core_change") and dt.itemsize == 24


def test_unknown_columns_raise_before_the_call():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQN")])
    args = (codes, offs, [0], [0, 0], [], [])
    for cols in (("core_score", "nosuch"), (), ("mw_score",)):
        with pytest.raises(ValueError, match="effect columns"):
            plaac_b200.Scorer.variant_effects(None, *args, columns=cols)  # (no ctx is needed to reject them)


def test_saturation_map_shape_order_and_nan():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MAX"), plaac_b200.encode(""), plaac_b200.encode("QN")])
    protein, first_sub, pos, code = plaac_b200.saturation(codes, offs)
    col = np.arange(len(protein), dtype=np.float64) + 0.5  # variant index + 0.5: each cell names its variant
    maps = plaac_b200.saturation_map(col, codes, offs)
    assert [m.shape for m in maps] == [(3, 20), (0, 20), (2, 20)]
    for p, m in zip((0, 2), (maps[0], maps[2])):
        ref = codes[offs[p]:offs[p + 1]]
        for i, r in enumerate(ref):
            for j, c in enumerate(range(1, 21)):  # columns A C D ... Y
                if c == r:
                    assert np.isnan(m[i, j])
                    continue
                v = int(m[i, j])
                assert protein[v] == p and first_sub[v + 1] - first_sub[v] == 1
                assert pos[first_sub[v]] == i and code[first_sub[v]] == c
    assert np.isnan(maps[0]).sum() == 2 and not np.isnan(maps[0][2]).any()  # M, A; X keeps all 20
    assert np.isnan(maps[2]).sum() == 2
    # a subset, in the order given
    pr, fs, ps, cs = plaac_b200.saturation(codes, offs, proteins=[2, 0])
    sub = plaac_b200.saturation_map(np.arange(len(pr), dtype=np.float64), codes, offs, proteins=[2, 0])
    assert [m.shape for m in sub] == [(2, 20), (3, 20)] and sub[1][0, 0] == 40  # QN: 1 + 38 rows, then MAX's WT
    with pytest.raises(ValueError):
        plaac_b200.saturation_map(col[:-1], codes, offs)
    with pytest.raises(ValueError):
        plaac_b200.saturation_map(np.r_[col, 0.0], codes, offs)


@pytest.fixture(scope="module")
def cli():
    pb.build_lib()
    path = pb.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args):
    return subprocess.run([cli, *args], capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("args, why", [
    (["--saturate", "--effects", "COREscore,Nope"], "unknown column 'Nope'"),
    (["--saturate", "--effects", "dLLR"], "unknown column 'dLLR'"),
    (["--saturate", "--effects", ""], "empty column name"),
    (["--saturate", "--effects", "LLR,"], "empty column name"),
    (["--effects", "LLR"], "--effects needs --variants FILE or --saturate"),
    (["--saturate", "--effects", "LLR", "-p", "all"], "cannot be combined with -p"),
    (["--saturate", "--effects", "LLR", "--rank"], "cannot be combined with --rank"),
    (["--saturate", "--effects", "LLR", "--gpus", "2"], "cannot be combined with --gpus > 1"),
    (["--variants", "VF", "--effects", "LLR", "-p", "all"], "cannot be combined with -p"),
])
def test_cli_effects_rejections(cli, tmp_path, args, why):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    vf = tmp_path / "v.txt"
    vf.write_text("a\tWT\n")
    r = run(cli, "-s", "-i", str(fa), *[str(vf) if a == "VF" else a for a in args])
    assert r.returncode == 2 and why in r.stderr, r.stderr
    assert r.stdout == ""


# ---------------------------------------------------------------------------------------------- GPU
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
    rec = scorer.score_variants(codes, offs, *var)
    return codes, offs, var, wt, rec


@pytest.fixture(scope="module")
def default_effects(scorer, case):
    codes, offs, var, wt, rec = case
    return scorer.variant_effects(codes, offs, *var, columns=plaac_b200.EFFECT_COLUMNS)


@pytest.mark.gpu
def test_effects_equal_the_subtraction(scorer, case, default_effects):
    codes, offs, var, wt, rec = case
    assert (wt["core_start"] >= 0).sum() > 5 and (rec["core_start"] >= 0).sum() > 20
    want = expected(rec, wt, var[0], plaac_b200.EFFECT_COLUMNS)
    cc = want["core_change"]
    assert (cc == -1).any() and (cc == 0).any()  # CORE lost and unchanged both occur
    assert np.isnan(want["llr"]).any() and np.isnan(want["core_score"]).any()
    assert_same_effects(default_effects, want, "all 14 columns")
    for k, n in enumerate(plaac_b200.EFFECT_COLUMNS):
        got = scorer.variant_effects(codes, offs, *var, columns=(n,))
        assert got.dtype.names == (n,)
        assert_same_effects(got, want[[n]], f"bit {k}")
    # the CORE change is the change of has_core
    assert np.array_equal(default_effects["core_change"],
                          np.isnan(wt["core_score"][var[0]]).astype(float) - np.isnan(rec["core_score"]).astype(float))
    # columns come back in bit order, whatever the order asked
    got = scorer.variant_effects(codes, offs, *var, columns=("core_change", "papa_llr2", "llr"))
    assert got.dtype.names == ("llr", "papa_llr2", "core_change")
    assert_same_effects(got, want[["llr", "papa_llr2", "core_change"]], "three columns")


@pytest.mark.gpu
def test_wild_records_equal_plaac_score(scorer, case):
    codes, offs, var, wt, rec = case
    eff, wild = scorer.variant_effects(codes, offs, *var, columns=("core_score",), wild=True)
    assert wild.dtype == plaac_b200.SUMMARY_DTYPE and len(wild) == len(offs) - 1
    assert wild.tobytes() == scorer.score(codes, offs).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["chunked", "pinned", "generic_windows", "kernel_variant_1", "long_fixed", "long_off",
                                 "long_auto"])
def test_other_code_paths(case, default_effects, how):
    codes, offs, var, wt, rec = case
    params = plaac_b200.default_params(ww1=31, ww2=41) if how == "generic_windows" else None
    sc = plaac_b200.Scorer(params)
    cols = plaac_b200.EFFECT_COLUMNS
    try:
        if how == "chunked":
            sc.set_chunk(0, 200)  # 15 chunks: every slot is reused many times
        elif how == "kernel_variant_1":
            sc.set_kernel_variant(1)
        elif how.startswith("long_"):
            sc.set_long_path({"long_fixed": 1024, "long_off": 0, "long_auto": -1}[how])
        if how == "pinned":
            with plaac_b200.PinnedBuffer(len(var[0]), dtype=plaac_b200.effects_dtype(ALL)) as buf:
                got = sc.variant_effects(codes, offs, *var, columns=cols, out=buf.array).copy()
        else:
            got = sc.variant_effects(codes, offs, *var, columns=cols)
        # (kernel variant 1 and other windows give records of their own; the effects are those records' differences)
        own = how in ("generic_windows", "kernel_variant_1")
        want = expected(sc.score_variants(codes, offs, *var), sc.score(codes, offs), var[0], cols) if own else default_effects
    finally:
        sc.close()
    assert_same_effects(got, want, how)


def _call(sc, codes, offs, nprot, protein, first_sub, pos, code, nvar, columns, eff, wild=None):
    V = plaac_b200.Variants(nvar=nvar, protein=protein, first_sub=first_sub, pos=pos, code=code)
    rc = plaac_b200.lib().plaac_score_variant_effects(sc._h, codes, offs, nprot, C.byref(V), columns, eff, wild)
    return rc, plaac_b200.lib().plaac_last_error(sc._h).decode()


def _call_records(sc, codes, offs, nprot, protein, first_sub, pos, code, nvar, out):
    V = plaac_b200.Variants(nvar=nvar, protein=protein, first_sub=first_sub, pos=pos, code=code)
    rc = plaac_b200.lib().plaac_score_variants(sc._h, codes, offs, nprot, C.byref(V), out)
    return rc, plaac_b200.lib().plaac_last_error(sc._h).decode()


@pytest.mark.gpu
def test_invalid_inputs_as_score_variants(scorer):
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDQQNKLLAPQ"), plaac_b200.encode("ACDEFG")])
    rec = np.zeros(8, dtype=plaac_b200.SUMMARY_DTYPE)
    eff = np.full(8 * 14, 7.0)
    arr = lambda a, t: np.ascontiguousarray(a, dtype=t)  # noqa: E731

    def ptrs(protein, first_sub, pos, code, null=()):
        a = [arr(protein, np.int32), arr(first_sub, np.int64), arr(pos, np.int32), arr(code, np.uint8)]
        return a, [None if i in null else x.ctypes.data for i, x in enumerate(a)]

    def both(*v, null=(), columns=ALL):
        a, p = ptrs(*v, null=null)
        r = _call_records(scorer, codes.ctypes.data, offs.ctypes.data, 2, *p, len(a[0]), rec.ctypes.data)
        e = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, *p, len(a[0]), columns, eff.ctypes.data)
        return r, e

    ok = ([0, 1], [0, 1, 2], [3, 5], [1, 2])
    r, e = both(*ok)
    assert r[0] == e[0] == 0
    cases = [([0, 2], [0, 1, 2], [3, 5], [1, 2]), ([-1, 1], [0, 1, 2], [3, 5], [1, 2]),
             ([0, 1], [0, 1, 2], [3, 6], [1, 2]), ([0, 1], [0, 1, 2], [-1, 5], [1, 2]),
             ([0, 1], [0, 2, 2], [3, 3], [1, 2]), ([0, 1], [0, 2, 2], [5, 3], [1, 2]),
             ([0, 1], [0, 1, 2], [3, 5], [1, 22]), ([0, 1], [1, 1, 2], [3, 5], [1, 2]),
             ([0, 1], [0, 2, 1], [3, 5], [1, 2])]
    for c in cases:
        r, e = both(*c)
        assert r[0] == -1 and e == r, (c, r, e)
    for k in range(4):
        r, e = both(*ok, null=(k,))
        assert r[0] == -1 and e == r, (k, r, e)
    # the effect call's own checks
    a, p = ptrs(*ok)
    for columns in (0, 1 << 14, -1):
        rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, *p, 2, columns, eff.ctypes.data)
        assert rc == -1 and "columns" in msg, (columns, msg)
    rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, *p, 2, ALL, None)
    assert rc == -1 and "NULL effects" in msg
    # nvar == 0: nothing written, not even the wild type
    eff[:] = 7.0
    wild = np.zeros(2, dtype=plaac_b200.SUMMARY_DTYPE)
    wild["llr"] = 7.0
    rc, _ = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, *p, 0, ALL, eff.ctypes.data, wild.ctypes.data)
    assert rc == 0 and (eff == 7.0).all() and (wild["llr"] == 7.0).all() and (wild["prot_len"] == 0).all()
    rc, _ = _call(scorer, codes.ctypes.data, offs.ctypes.data, 2, None, None, None, None, 0, ALL, None)
    assert rc == 0
    with pytest.raises(plaac_b200.PlaacError, match="variant 0: position 99"):
        scorer.variant_effects(codes, offs, [0], [0, 1], [99], [1])


@pytest.mark.gpu
def test_invalid_reference_bytes_every_effect_written(scorer):
    codes, offs = reference_batch()
    codes = codes.copy()
    codes[offs[3] + 1] = 30
    codes[offs[50] + 7] = 200
    wt = np.zeros(len(offs) - 1, dtype=plaac_b200.SUMMARY_DTYPE)
    rc_wt = plaac_b200.lib().plaac_score(scorer._h, codes.ctypes.data, offs.ctypes.data, len(offs) - 1, wt.ctypes.data, None)
    var = [np.ascontiguousarray(x) for x in build_variants(codes, offs, wt, 600, seed=9)]
    rec = np.zeros(len(var[0]), dtype=plaac_b200.SUMMARY_DTYPE)
    rc_rec, _ = _call_records(scorer, codes.ctypes.data, offs.ctypes.data, len(offs) - 1, *[x.ctypes.data for x in var],
                              len(var[0]), rec.ctypes.data)
    want = expected(rec, wt, var[0], plaac_b200.EFFECT_COLUMNS)
    # variants on the clean proteins only, so that the error can come from the reference's own records alone
    clean = np.nonzero(~np.isin(var[0], [3, 50]))[0]
    for sel in (np.arange(len(var[0])), clean):
        protein = np.ascontiguousarray(var[0][sel])
        nsub = np.diff(var[1])[sel]
        first_sub = np.r_[0, np.cumsum(nsub)].astype(np.int64)
        take = np.concatenate([np.arange(var[1][v], var[1][v + 1]) for v in sel]).astype(np.int64)
        pos, code = np.ascontiguousarray(var[2][take]), np.ascontiguousarray(var[3][take])
        got = np.full(len(sel), np.inf, dtype=plaac_b200.effects_dtype(ALL))
        wild = np.zeros(len(offs) - 1, dtype=plaac_b200.SUMMARY_DTYPE)
        rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, len(offs) - 1, protein.ctypes.data, first_sub.ctypes.data,
                        pos.ctypes.data, code.ctypes.data, len(sel), ALL, got.ctypes.data, wild.ctypes.data)
        assert rc_wt == -1 and rc_rec == -1 and rc == -1 and "> 21" in msg, msg
        assert wild.tobytes() == wt.tobytes()
        assert_same_effects(got, want[sel], f"invalid reference bytes, {len(sel)} variants")


@pytest.mark.gpu
def test_saturation_of_the_classic_prions(scorer, golden):
    """core_change and dCOREscore of the scan equal those of the records test_variants checks against the oracle."""
    seqs = [plaac_b200.encode(p["seq"]) for p in golden["proteins"]]
    codes, offs = plaac_b200.pack(seqs)
    var = plaac_b200.saturation(codes, offs)
    rec = scorer.score_variants(codes, offs, *var)
    wt = scorer.score(codes, offs)
    got = scorer.variant_effects(codes, offs, *var, columns=("core_score", "core_change"))
    assert_same_effects(got, expected(rec, wt, var[0], ("core_score", "core_change")), "classic prions")
    assert np.isin(got["core_change"], [-1.0, 0.0, 1.0]).all()
    maps = plaac_b200.saturation_map(got["core_score"], codes, offs)
    assert [m.shape for m in maps] == [(len(s), 20) for s in seqs]
    for s, m in zip(seqs, maps):
        i = np.nonzero((s >= 1) & (s <= 20))[0]
        assert np.isnan(m[i, s[i] - 1]).all() and np.isnan(m).sum() == len(i)


def _fasta(names, seqs):
    return "".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in zip(names, seqs))


@pytest.mark.gpu
def test_cli_effects_match_the_api(cli, scorer, tmp_path, golden):
    rng = np.random.default_rng(23)
    names = [p["name"] for p in golden["proteins"][:2]] + ["rand1"]
    seqs = [p["seq"].rstrip("*") for p in golden["proteins"][:2]] + ["".join(AA[c] for c in rng.integers(1, 21, 90))]
    fa = tmp_path / "small.fa"
    fa.write_text(_fasta(names, seqs))
    codes, offs = plaac_b200.pack([plaac_b200.encode(s) for s in seqs])
    s0, s2 = seqs[0], seqs[2]
    lines = [(names[2], f"{s2[0]}1P"), (names[0], "WT"), (names[2], f"{s2[5]}6Q,{s2[1]}2N"), (names[0], f"{s0[9]}10X"),
             (names[0], f"{s0[0]}1A,{s0[-1]}{len(s0)}P"), (names[0], f"{s0[19]}20*")]
    vf = tmp_path / "v.txt"
    vf.write_text("".join(f"{n}\t{sp}\n" for n, sp in lines))
    # the variants in the CLI's row order: record order, then file order
    protein, first_sub, pos, code = [], [0], [], []
    for rec in range(len(names)):
        for n, sp in lines:
            if n != names[rec]:
                continue
            subs = [] if sp == "WT" else sorted((int(t[1:-1]) - 1, AA.index(t[-1])) for t in sp.split(","))
            protein.append(rec)
            pos += [q for q, _ in subs]
            code += [c for _, c in subs]
            first_sub.append(len(pos))
    mode_var = (["--variants", str(vf)], "COREscore,LLR,COREchange", ("core_score", "llr", "core_change"),
                (protein, first_sub, pos, code))
    mode_sat = (["--saturate"], "PRDscore", ("prd_score",), plaac_b200.saturation(codes, offs))
    for mode, cols, py_cols, var in (mode_var, mode_sat):
        a = run(cli, "-s", "-i", str(fa), *mode, "--effects", cols)
        b = run(cli, "-s", "-i", str(fa), *mode)
        assert a.returncode == 0 and b.returncode == 0, a.stderr + b.stderr
        al = a.stdout.rstrip("\n").split("\n")
        bl = b.stdout.rstrip("\n").split("\n")
        want_head = ["SEQid"] + [("" if c == "COREchange" else "d") + c
                                 for c in sorted(cols.split(","), key=CLI_NAMES.index)]
        assert al[0].split("\t") == want_head
        assert [x.split("\t")[0] for x in al[1:]] == [x.split("\t")[0] for x in bl[1:]]
        eff = scorer.variant_effects(codes, offs, *var, columns=py_cols)
        assert len(al) - 1 == len(eff) > 5
        for line, e in zip(al[1:], eff):
            cells = line.split("\t")[1:]
            want = [str(int(e[n])) if n == "core_change" else java_fmt(e[n], 3) for n in eff.dtype.names]
            assert cells == want, (line, want)
    # the parameter block is printed unless -s
    a = run(cli, "-i", str(fa), "--saturate", "--effects", "LLR")
    assert a.returncode == 0 and a.stdout.startswith("####") and "\nSEQid\tdLLR\n" in a.stdout
