"""Shuffled replicates (plaac_shuffle_host, plaac_score_shuffles, Scorer.shuffle_null, the CLI's --null).

Replicate r of protein i is a permutation of its residues that DESIGN.md section 13 defines; `restate` below is that
text in numpy.  A replicate's values are, bit for bit, the record plaac_score gives for the materialised replicate, so
the oracle of every GPU test here is plaac_score on a batch built with plaac_shuffle_host, and the counting rule applied
in numpy."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import plaac_b200
from oracle import orc
from tests import parity, synth
from tests.test_variants import reference_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NT = max(1, min(32, os.cpu_count() or 1))
AA = "XACDEFGHIKLMNPQRSTVWY*"
ALL = (1 << 14) - 1
NAMES = plaac_b200.NULL_COLUMNS
CLI_NAMES = ["LLR", "COREscore", "PRDscore", "HMMall", "HMMvit", "FImeanhydro", "FImeancharge", "FImeancombo",
             "PAPAcombo", "PAPAprop", "PAPAfi", "PAPAllr", "PAPAllr2", "hasCORE"]
M64 = (1 << 64) - 1
GAMMA = 0x9E3779B97F4A7C15


# ---------------------------------------------------------------------------------------------- helpers
def _mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return z ^ (z >> 31)


def _mix32(x):
    x = x.astype(np.uint64)
    x ^= x >> np.uint64(16)
    x = (x * np.uint64(0x7FEB352D)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(15)
    x = (x * np.uint64(0x846CA68B)) & np.uint64(0xFFFFFFFF)
    x ^= x >> np.uint64(16)
    return x


def restate(n, seed, protein, replicate, t=None):
    """pi(t) as DESIGN.md section 13 writes it (for t = 0..n-1 unless given)."""
    t = np.arange(n, dtype=np.uint64) if t is None else np.asarray(t, dtype=np.uint64)
    if n <= 1:
        return t
    b = int(n - 1).bit_length()
    s = _mix64((seed + GAMMA) & M64) ^ protein
    s = _mix64((s + GAMMA) & M64) ^ replicate
    keys = [_mix64((s + (k + 1) * GAMMA) & M64) & 0xFFFFFFFF for k in range(6)]

    def feistel(x):
        for k in range(6):
            w = b // 2 if k % 2 == 0 else b - b // 2
            R = x & np.uint64((1 << w) - 1)
            L = x >> np.uint64(w)
            F = _mix32(R ^ np.uint64(keys[k])) & np.uint64((1 << (b - w)) - 1)
            x = (R << np.uint64(b - w)) | (L ^ F)
        return x

    y = feistel(t.copy())
    while True:
        m = y >= n
        if not m.any():
            return y
        y[m] = feistel(y[m])


def host_perm(n, seed, protein, replicate):
    """pi through plaac_shuffle_host: shuffle the identity (as uint8 digits, so n <= 256 -- or several digit planes)."""
    idx = np.arange(n, dtype=np.int64)
    out = np.zeros(n, dtype=np.int64)
    for plane in range(4):
        digits = ((idx >> (8 * plane)) & 255).astype(np.uint8)
        rep = np.empty(n, dtype=np.uint8)
        rc = plaac_b200.lib().plaac_shuffle_host(digits.ctypes.data, n, seed, protein, replicate, rep.ctypes.data)
        assert rc == 0
        out |= rep.astype(np.int64) << (8 * plane)
        if n <= 256 << (8 * plane):
            break
    return out


def materialise(codes, offs, K, seed, proteins):
    """Every replicate, row j*K + r = replicate r of protein proteins[j], as one ordinary batch."""
    seqs = [plaac_b200.shuffle(codes, offs, int(i), r, seed) for i in proteins for r in range(K)]
    return plaac_b200.pack(seqs)


def key(x):
    return np.where(np.isnan(x), -np.inf, x)


def expected_counts(rec, obs, K, names):
    """The counting rule of the contract, in numpy: rec has nsel*K rows, obs nsel."""
    nsel = len(obs)
    out = np.zeros(nsel, dtype=[(n, "<i8") for n in names])
    for n in names:
        if n == "has_core":
            hit = ~np.isnan(rec["core_score"])
        else:
            hit = key(rec[n]).reshape(nsel, K) >= key(obs[n])[:, None]
        out[n] = hit.reshape(nsel, K).sum(axis=1)
    return out


def values_of(rec, names):
    out = np.zeros(len(rec), dtype=[(n, "<f8") for n in names])
    for n in names:
        out[n] = (~np.isnan(rec["core_score"])).astype(np.float64) if n == "has_core" else rec[n]
    return out


def assert_same_values(got, want, what):
    """Bitwise, with every NaN equal to every other NaN."""
    assert got.dtype.names == want.dtype.names, what
    for n in want.dtype.names:
        g, w = np.ascontiguousarray(got[n]).ravel(), np.ascontiguousarray(want[n]).ravel()
        gn, wn = np.isnan(g), np.isnan(w)
        bad = np.nonzero((gn != wn) | (~gn & (g.view(np.uint64) != w.view(np.uint64))))[0]
        assert len(bad) == 0, f"{what}, {n}: {len(bad)} of {len(g)} differ, first {bad[:10].tolist()}"


# ---------------------------------------------------------------------------------------------- CPU: the shuffle
def test_bijection_and_composition_small_and_around_2_16():
    rng = np.random.default_rng(1)
    for n in list(range(0, 301)) + [(1 << 16) - 1, 1 << 16, (1 << 16) + 1]:
        for protein, replicate in ((0, 0), (int(rng.integers(0, 1 << 30)), int(rng.integers(0, 1 << 20)))):
            p = host_perm(n, 12345, protein, replicate)
            assert np.array_equal(np.sort(p), np.arange(n)), n
            codes = rng.integers(0, 256, n).astype(np.uint8)  # bytes > 21 move like any other byte
            rep = np.empty(n, dtype=np.uint8)
            assert plaac_b200.lib().plaac_shuffle_host(codes.ctypes.data, n, 12345, protein, replicate, rep.ctypes.data) == 0
            assert np.array_equal(rep, codes[p])
            assert np.array_equal(np.bincount(rep, minlength=256), np.bincount(codes, minlength=256))


@pytest.mark.parametrize("n", [10**6, 2**31 - 1])
def test_bijection_on_sampled_positions_of_large_n(n):
    t = np.random.default_rng(n % 997).choice(n, 100000, replace=False)
    img = restate(n, 99, 7, 3, t)
    assert (img < n).all() and len(np.unique(img)) == len(t)
    if n == 10**6:
        assert np.array_equal(host_perm(n, 99, 7, 3)[t], img.astype(np.int64))


def test_restatement_equals_plaac_shuffle_host():
    rng = np.random.default_rng(2)
    cases = [(n, int(rng.integers(0, 1 << 63)) * 2 + int(rng.integers(0, 2)), int(rng.integers(0, 1 << 31)),
              int(rng.integers(0, 1 << 40))) for n in (2, 3, 4, 5, 7, 8, 9, 33, 64, 65, 255, 256, 257, 1000, 4097, 34000)]
    cases += [(int(rng.integers(2, 70000)), int(rng.integers(0, 1 << 62)), int(rng.integers(0, 100)), r) for r in range(60)]
    for n, seed, protein, replicate in cases:
        assert np.array_equal(host_perm(n, seed, protein, replicate), restate(n, seed, protein, replicate).astype(np.int64)), \
            (n, seed, protein, replicate)
    # n <= 1 is the identity
    assert restate(1, 5, 5, 5).tolist() == [0] and host_perm(1, 5, 5, 5).tolist() == [0]


def test_python_shuffle_wraps_the_host_function():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDAAKLR"), plaac_b200.encode(""), plaac_b200.encode("QNYQ")])
    for i in range(3):
        s = codes[offs[i]:offs[i + 1]]
        assert np.array_equal(plaac_b200.shuffle(codes, offs, i, 4, seed=17), s[restate(len(s), 17, i, 4).astype(np.int64)])
    with pytest.raises(plaac_b200.PlaacError, match="negative"):
        plaac_b200.shuffle(codes, offs, 0, -1)


def test_quality_all_permutations_of_three():
    perms = {}
    for r in range(60000):
        p = tuple(host_perm(3, 2024, 11, r))
        perms[p] = perms.get(p, 0) + 1
    assert len(perms) == 6
    f = np.array(list(perms.values()), dtype=np.float64)
    chi2 = ((f - 10000.0) ** 2 / 10000.0).sum()
    assert chi2 < stats.chi2.isf(1e-6, 5), (chi2, perms)


def test_quality_positions_uniform_and_one_fixed_point_at_61():
    N, n = 6000, 61
    T = np.zeros((n, n))
    fixed = 0
    for r in range(N):
        p = restate(n, 31, 5, r).astype(np.int64)
        T[np.arange(n), p] += 1
        fixed += int((p == np.arange(n)).sum())
    E = N / n
    chi2 = ((T - E) ** 2 / E).sum()
    assert chi2 < stats.chi2.isf(1e-6, n * (n - 1)), chi2
    # fixed points of a uniform permutation: mean 1, variance 1
    assert abs(fixed / N - 1.0) < 5.0 / np.sqrt(N), fixed / N


def test_quality_replicates_differ():
    for n in (20, 61, 300):
        seen = {tuple(restate(n, 8, 3, r)) for r in range(2000)}
        assert len(seen) == 2000, n
    # seeds and proteins select different permutations too
    assert len({tuple(restate(50, s, p, 0)) for s in range(30) for p in range(30)}) == 900


# ---------------------------------------------------------------------------------------------- CPU: interfaces
def test_null_struct_and_bits_match_the_header(tmp_path):
    src = tmp_path / "n.c"
    fields = ["replicates", "seed", "columns", "reserved", "nsel", "proteins", "counts", "values"]
    src.write_text('#include <stddef.h>\n#include <stdio.h>\n#include "plaac_cuda.h"\nint main(void){'
                   'printf("%zu %d %d\\n", sizeof(plaac_null), PLAAC_NULL_HAS_CORE, PLAAC_EFFECT_PAPA_LLR2);'
                   + "".join(f'printf("%zu\\n", offsetof(plaac_null, {f}));' for f in fields) + "return 0;}\n")
    exe = tmp_path / "n"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[:3] == [C.sizeof(plaac_b200.Null), 1 << 13, 1 << 12]
    assert got[3:] == [getattr(plaac_b200.Null, f).offset for f in fields]
    assert NAMES[:13] == plaac_b200.EFFECT_COLUMNS[:13] and NAMES[13] == "has_core"


def test_unknown_columns_raise_before_the_call():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQN")])
    for cols in (("core_score", "nosuch"), (), ("core_change",), ("mw_score",)):
        with pytest.raises(ValueError, match="null columns"):
            plaac_b200.Scorer.shuffle_null(None, codes, offs, 5, columns=cols)  # (no ctx is needed to reject them)


@pytest.fixture(scope="module")
def cli():
    from plaac_b200 import build as pb

    pb.build_lib()
    path = pb.build_cli()
    assert path and os.path.exists(path)
    return path


def run(cli, *args):
    return subprocess.run([cli, *args], capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("args, why", [
    (["--null", "NF", "--replicates", "5", "-p", "all"], "cannot be combined with -p"),
    (["--null", "NF", "--replicates", "5", "--saturate"], "cannot be combined with --saturate"),
    (["--null", "NF", "--replicates", "5", "--variants", "VF"], "cannot be combined with --variants"),
    (["--null", "NF", "--replicates", "5", "--segments", "SF"], "cannot be combined with --segments"),
    (["--null", "NF", "--replicates", "5", "--gpu-ingest"], "cannot be combined with --gpu-ingest"),
    (["--null", "NF", "--replicates", "5", "--gpus", "2"], "cannot be combined with --gpus > 1"),
    (["--null", "NF"], "--replicates"),
    (["--null", "NF", "--replicates", "0"], "--replicates"),
    (["--null", "NF", "--replicates", "-3"], "--replicates"),
    (["--replicates", "5"], "needs --null"),
    (["--seed", "5"], "needs --null"),
    (["--null-columns", "LLR"], "needs --null"),
    (["--null", "NF", "--replicates", "5", "--null-columns", "LLR,Nope"], "unknown column 'Nope'"),
    (["--null", "NF", "--replicates", "5", "--null-columns", "COREchange"], "unknown column 'COREchange'"),
    (["--null", "NF", "--replicates", "5", "--null-columns", ""], "empty column name"),
])
def test_cli_null_rejections(cli, tmp_path, args, why):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    vf = tmp_path / "v.txt"
    vf.write_text("a\tWT\n")
    files = {"VF": str(vf), "NF": str(tmp_path / "null.txt"), "SF": str(tmp_path / "seg.txt")}
    r = run(cli, "-s", "-i", str(fa), *[files.get(a, a) for a in args])
    assert r.returncode == 2 and why in r.stderr, r.stderr
    assert r.stdout == ""


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def scorer():
    s = plaac_b200.Scorer()
    yield s
    s.close()


def null_batch(golden):
    """Classic prions, synthetic and repeat proteins, and the edge cases: empty proteins, length 1, shorter than the
    core."""
    parts = [plaac_b200.pack([plaac_b200.encode(p["seq"]) for p in golden["proteins"]]), synth.edge_cases(),
             synth.proteome(60, seed=44), synth.repeat_proteome(30, seed=45)]
    seqs = []
    for c, o in parts:
        seqs += [c[o[i]:o[i + 1]] for i in range(len(o) - 1)]
    seqs += [np.zeros(0, dtype=np.uint8), np.array([14], dtype=np.uint8), plaac_b200.encode("QNQNQYQQ" * 5)]
    return plaac_b200.pack(seqs)


@pytest.fixture(scope="module")
def case(scorer, golden):
    codes, offs = null_batch(golden)
    K, seed = 64, 1234
    nprot = len(offs) - 1
    counts, vals, obs = scorer.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, values=True, observed=True)
    mc, mo = materialise(codes, offs, K, seed, range(nprot))
    rec = scorer.score(mc, mo)
    return codes, offs, K, seed, counts, vals, obs, rec


@pytest.mark.gpu
def test_exact_against_the_materialised_replicates(scorer, case):
    codes, offs, K, seed, counts, vals, obs, rec = case
    nprot = len(offs) - 1
    lens = np.diff(offs)
    assert (lens == 0).any() and (lens == 1).any() and ((lens > 1) & (lens < 60)).any() and lens.max() > 1000
    assert obs.tobytes() == scorer.score(codes, offs).tobytes()
    assert vals.shape == (nprot, K)
    assert_same_values(vals.reshape(-1), values_of(rec, NAMES), "values")
    want = expected_counts(rec, obs, K, NAMES)
    for n in NAMES:
        assert np.array_equal(counts[n], want[n]), n
    # the data exercise the rule: both ends of the range, NaN observed CORE, -Inf LLR
    c = counts["core_score"]
    assert (c == 0).any() and (c == K).any() and ((c > 0) & (c < K)).any()
    assert np.isnan(obs["core_score"]).any() and np.isneginf(obs["llr"]).any()
    # a few columns alone, and in any order
    got = scorer.shuffle_null(codes, offs, K, seed=seed, columns=("hmm_all", "papa_fi", "has_core"))
    assert got.dtype.names == ("hmm_all", "papa_fi", "has_core")
    for n in got.dtype.names:
        assert np.array_equal(got[n], want[n]), n
    # the default columns
    got = scorer.shuffle_null(codes, offs, K, seed=seed)
    assert got.dtype.names == ("llr", "core_score", "hmm_all")
    assert all(np.array_equal(got[n], want[n]) for n in got.dtype.names)


@pytest.mark.gpu
def test_values_agree_with_the_oracle(case):
    codes, offs, K, seed, counts, vals, obs, rec = case
    rng = np.random.default_rng(3)
    rows = np.sort(rng.choice(len(rec), 3000, replace=False))
    nprot = len(offs) - 1
    seqs = [plaac_b200.shuffle(codes, offs, int(q // K), int(q % K), seed) for q in rows]
    mc, mo = plaac_b200.pack(seqs)
    P = orc.make_params()
    ref = orc.score_batch(P, mc, mo, nthreads=NT)
    got = rec[rows].copy()
    bad, nties = parity.compare_with_tie_classes(P, mc, mo, got, ref, orc.INT_FIELDS, orc.DBL_FIELDS)
    assert not bad, "\n".join(bad[:20])
    assert nties <= len(rows) // 100
    assert_same_values(vals.reshape(-1)[rows], values_of(rec[rows], NAMES), "sampled values")
    assert nprot > 0


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["chunked", "long_fixed", "long_off", "long_auto", "kernel_variant_1", "generic_windows",
                                 "pinned", "subset"])
def test_invariance(case, how):
    codes, offs, K, seed, counts, vals, obs, rec = case
    params = plaac_b200.default_params(ww1=31, ww2=41) if how == "generic_windows" else None
    sc = plaac_b200.Scorer(params)
    nprot = len(offs) - 1
    try:
        if how == "chunked":
            sc.set_chunk(0, 300)  # many chunks that cut proteins' replicate runs
        elif how == "kernel_variant_1":
            sc.set_kernel_variant(1)
        elif how.startswith("long_"):
            sc.set_long_path({"long_fixed": 1024, "long_off": 0, "long_auto": -1}[how])
        if how == "subset":
            sel = np.array([5, 0, nprot - 1, 5, 17, 2, nprot - 3], dtype=np.int32)
            c, v, o = sc.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, proteins=sel, values=True, observed=True)
            for n in NAMES:
                assert np.array_equal(c[n], counts[n][sel]), n
            assert_same_values(v, vals[sel], "subset values")
            assert o.tobytes() == obs[sel].tobytes()
            return
        if how == "pinned":
            nl = plaac_b200.Null(replicates=K, seed=seed, columns=ALL, reserved=0, nsel=-1, proteins=None)
            with plaac_b200.PinnedBuffer(nprot, dtype=counts.dtype) as cb, \
                    plaac_b200.PinnedBuffer(nprot * K, dtype=vals.dtype) as vb, \
                    plaac_b200.PinnedBuffer(nprot, dtype=plaac_b200.SUMMARY_DTYPE) as ob:
                nl.counts, nl.values = cb.array.ctypes.data, vb.array.ctypes.data
                rc = plaac_b200.lib().plaac_score_shuffles(sc._h, codes.ctypes.data, offs.ctypes.data, nprot, C.byref(nl),
                                                           ob.array.ctypes.data)
                assert rc == 0
                c, v, o = cb.array.copy(), vb.array.copy().reshape(nprot, K), ob.array.copy()
            assert o.tobytes() == obs.tobytes()
        else:
            c, v = sc.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, values=True)
        if how in ("generic_windows", "kernel_variant_1"):
            # other windows (and kernel variant 1) give records of their own: compare with those of the same ctx
            mc, mo = materialise(codes, offs, K, seed, range(nprot))
            r2 = sc.score(mc, mo)
            want_c, want_v = expected_counts(r2, sc.score(codes, offs), K, NAMES), values_of(r2, NAMES).reshape(nprot, K)
        else:
            want_c, want_v = counts, vals
    finally:
        sc.close()
    for n in NAMES:
        assert np.array_equal(c[n], want_c[n]), (how, n)
    assert_same_values(v, want_v, how)


@pytest.mark.gpu
def test_long_protein_replicates(scorer):
    codes, offs = synth.long_proteins(seed=47, lengths=(34000,))
    K, seed = 8, 77
    for thr in (-1, 1024):
        scorer.set_long_path(thr)
        try:
            c, v, o = scorer.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, values=True, observed=True)
        finally:
            scorer.set_long_path(-1)
        mc, mo = materialise(codes, offs, K, seed, [0])
        rec = scorer.score(mc, mo)
        assert_same_values(v.reshape(-1), values_of(rec, NAMES), f"34 000 residues, threshold {thr}")
        want = expected_counts(rec, o, K, NAMES)
        assert all(np.array_equal(c[n], want[n]) for n in NAMES)


@pytest.mark.gpu
def test_more_than_2_31_replicate_residues(scorer):
    """A yeast-sized reference x K = 1000: sampled proteins against the materialised check, counts against values."""
    codes, offs = synth.proteome(6000, seed=48)
    K, seed = 1000, 5
    lens = np.diff(offs)
    assert int(lens.sum()) * K > 2**31
    cols = ("llr", "core_score", "has_core")
    c, v, o = scorer.shuffle_null(codes, offs, K, seed=seed, columns=cols, values=True, observed=True)
    for n in cols:
        if n == "has_core":
            assert np.array_equal(c[n], (v[n] == 1.0).sum(axis=1))
        else:
            assert np.array_equal(c[n], (key(v[n]) >= key(o[n])[:, None]).sum(axis=1)), n
    rng = np.random.default_rng(4)
    last = len(lens) - 1
    pick = [0, last] + rng.choice(len(lens), 4, replace=False).tolist()
    for i in pick:
        mc, mo = materialise(codes, offs, K, seed, [i])
        rec = scorer.score(mc, mo)
        assert_same_values(v[i], values_of(rec, cols), f"protein {i}")


def _call(sc, codes, offs, nprot, K, columns, nsel, proteins, counts, values=None, observed=None, reserved=0, seed=0):
    nl = plaac_b200.Null(replicates=K, seed=seed, columns=columns, reserved=reserved, nsel=nsel, proteins=proteins,
                         counts=counts, values=values)
    rc = plaac_b200.lib().plaac_score_shuffles(sc._h, codes, offs, nprot, C.byref(nl), observed)
    return rc, plaac_b200.lib().plaac_last_error(sc._h).decode()


@pytest.mark.gpu
def test_errors_and_edges(scorer):
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDQQNKLLAPQ"), plaac_b200.encode("ACDEFG")])
    cp, op = codes.ctypes.data, offs.ctypes.data
    sel = np.array([1, 0], dtype=np.int32)
    cnt = np.full(2 * 14, 7, dtype=np.int64)
    for kw, what in [(dict(K=-1), "replicates -1"), (dict(nsel=-2), "nsel -2"), (dict(reserved=1), "reserved"),
                     (dict(columns=0), "columns"), (dict(columns=1 << 14), "columns"), (dict(columns=-1), "columns"),
                     (dict(proteins=None), "NULL proteins"), (dict(counts=None), "NULL counts"),
                     (dict(nsel=-1, counts=None), "NULL counts")]:
        a = dict(K=4, columns=ALL, nsel=2, proteins=sel.ctypes.data, counts=cnt.ctypes.data)
        a.update(kw)
        rc, msg = _call(scorer, cp, op, 2, a["K"], a["columns"], a["nsel"], a["proteins"], a["counts"],
                        reserved=a.get("reserved", 0))
        assert rc == -1 and what in msg, (kw, msg)
    for bad in ([0, 2], [-1, 0], [1, 1, 0, 5]):
        b = np.array(bad, dtype=np.int32)
        j = next(k for k, x in enumerate(bad) if not 0 <= x < 2)
        rc, msg = _call(scorer, cp, op, 2, 4, ALL, len(b), b.ctypes.data, cnt.ctypes.data)
        assert rc == -1 and f"selected protein {j}: index {bad[j]}" in msg, msg
    # K == 0: counts are 0 and observed is written
    obs = np.zeros(2, dtype=plaac_b200.SUMMARY_DTYPE)
    rc, _ = _call(scorer, cp, op, 2, 0, ALL, 2, sel.ctypes.data, cnt.ctypes.data, observed=obs.ctypes.data)
    assert rc == 0 and (cnt[:28] == 0).all() and obs.tobytes() == scorer.score(codes, offs)[sel].tobytes()
    # nsel == 0 and nprot == 0: PLAAC_OK, nothing written
    cnt[:] = 7
    rc, _ = _call(scorer, cp, op, 2, 4, ALL, 0, sel.ctypes.data, None)
    assert rc == 0
    rc, _ = _call(scorer, cp, op, 0, 4, ALL, -1, None, None)
    assert rc == 0 and (cnt == 7).all()
    c = scorer.shuffle_null(codes, offs, 3, proteins=[])
    assert len(c) == 0


@pytest.mark.gpu
def test_invalid_reference_bytes_everything_written(scorer):
    codes, offs = reference_batch()
    codes = codes.copy()
    codes[offs[3] + 1] = 30
    codes[offs[50] + 7] = 200
    nprot = len(offs) - 1
    K, seed = 5, 3
    sel = np.array([3, 50, 7, 3], dtype=np.int32)
    counts = np.full(len(sel), -1, dtype=[(n, "<i8") for n in NAMES])
    vals = np.full((len(sel), K), np.inf, dtype=[(n, "<f8") for n in NAMES])
    obs = np.zeros(len(sel), dtype=plaac_b200.SUMMARY_DTYPE)
    rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, nprot, K, ALL, len(sel), sel.ctypes.data,
                    counts.ctypes.data, vals.ctypes.data, obs.ctypes.data, seed=seed)
    assert rc == -1 and "> 21" in msg, msg
    wt = np.zeros(nprot, dtype=plaac_b200.SUMMARY_DTYPE)
    assert plaac_b200.lib().plaac_score(scorer._h, codes.ctypes.data, offs.ctypes.data, nprot, wt.ctypes.data, None) == -1
    assert obs.tobytes() == wt[sel].tobytes()
    mc, mo = materialise(codes, offs, K, seed, sel)
    rec = np.zeros(len(mo) - 1, dtype=plaac_b200.SUMMARY_DTYPE)
    plaac_b200.lib().plaac_score(scorer._h, mc.ctypes.data, mo.ctypes.data, len(mo) - 1, rec.ctypes.data, None)
    assert_same_values(vals.reshape(-1), values_of(rec, NAMES), "values with bytes > 21")
    want = expected_counts(rec, obs, K, NAMES)
    assert all(np.array_equal(counts[n], want[n]) for n in NAMES)


def _fasta(names, seqs):
    return "".join(f">{n}\n" + "".join(s[i:i + 60] + "\n" for i in range(0, len(s), 60)) for n, s in zip(names, seqs))


@pytest.mark.gpu
def test_cli_null_file_matches_the_api(cli, scorer, tmp_path, golden):
    rng = np.random.default_rng(29)
    names = [p["name"] for p in golden["proteins"]] + ["rand1", "short"]
    seqs = [p["seq"].rstrip("*") for p in golden["proteins"]] + ["".join(AA[c] for c in rng.integers(1, 21, 300)), "QNQ"]
    fa = tmp_path / "small.fa"
    fa.write_text(_fasta(names, seqs))
    codes, offs = plaac_b200.pack([plaac_b200.encode(s) for s in seqs])
    K = 50
    plain = run(cli, "-s", "-i", str(fa))
    assert plain.returncode == 0, plain.stderr
    outs = {}
    for tag, extra in (("default", []), ("cols", ["--null-columns", "hasCORE,PAPAcombo,LLR"]), ("seed", ["--seed", "9"]),
                       ("seed_again", ["--seed", "9"])):
        nf = tmp_path / f"null_{tag}.txt"
        r = run(cli, "-s", "-i", str(fa), "--null", str(nf), "--replicates", str(K), *extra)
        assert r.returncode == 0, r.stderr
        assert r.stdout == plain.stdout, tag
        outs[tag] = nf.read_text()
    assert outs["seed"] == outs["seed_again"] and outs["seed"] != outs["default"]
    for tag, seed, cols in (("default", 0, ("llr", "core_score", "hmm_all")),
                            ("cols", 0, ("llr", "papa_combo", "has_core")), ("seed", 9, ("llr", "core_score", "hmm_all"))):
        lines = outs[tag].rstrip("\n").split("\n")
        head = ["SEQid", "NULLreps"]
        for n in cols:
            cn = CLI_NAMES[NAMES.index(n)]
            head += [f"n{cn}"] + ([] if n == "has_core" else [f"p{cn}"])
        assert lines[0].split("\t") == head, tag
        # the rows follow the records the CLI prints (stdout), in that order
        printed = [x.split("\t")[0] for x in plain.stdout.rstrip("\n").split("\n")[1:]]
        assert [x.split("\t")[0] for x in lines[1:]] == printed
        want = scorer.shuffle_null(codes, offs, K, seed=seed, columns=cols)
        row = {nm: i for i, nm in enumerate(names)}
        for line in lines[1:]:
            cells = line.split("\t")
            j = row[cells[0]]
            assert cells[1] == str(K)
            exp = []
            for n in cols:
                exp.append(str(int(want[n][j])))
                if n != "has_core":
                    exp.append("%.6g" % ((1 + int(want[n][j])) / (1 + K)))
            assert cells[2:] == exp, (tag, line, exp)
