"""Sequential shuffle nulls (plaac_score_shuffles_seq, Scorer.shuffle_null_seq, seq_pvalues, the CLI's --stop-hits).

The oracle of every GPU test here is the fixed call itself: shuffle_null(..., K = K_max, values=True), whose values
tests/test_shuffle_null.py pins against materialised replicates and the CPU oracle.  `restate` turns those values into
the expected count and L of the contract (include/plaac_cuda.h, DESIGN.md section 14): the cumulative sum of the hits,
the first replicate where it reaches h, K_max where it never does."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plaac_b200
from tests import synth
from tests.test_shuffle_null import ALL, CLI_NAMES, NAMES, _fasta, key, null_batch
from tests.test_variants import reference_batch

DEFAULT = ("llr", "core_score", "hmm_all")


def hits_of(vals, obs, n):
    """Replicate hits of column n: vals (nsel, K) of the fixed call, obs the observed records."""
    if n == "has_core":
        return vals[n] == 1.0
    return key(vals[n]) >= key(obs[n])[:, None]


def restate(vals, obs, names, h, K):
    """count and L of the contract, from the first K replicates' values."""
    nsel = len(obs)
    counts = np.zeros(nsel, dtype=[(n, "<i8") for n in names])
    scored = np.zeros(nsel, dtype=counts.dtype)
    if K == 0:
        return counts, scored
    for n in names:
        cs = np.cumsum(hits_of(vals, obs, n)[:, :K], axis=1)
        stopped = cs[:, -1] >= h
        counts[n] = np.where(stopped, h, cs[:, -1])
        scored[n] = np.where(stopped, np.argmax(cs >= h, axis=1) + 1, K)
    return counts, scored


CHUNK_RES = 256 << 20  # the library's default chunk bound
SMALL = 1 << 20  # a chunk bound that makes the rounds here short: many rounds


def bounds(lens, scored, h, K, chunk_res=CHUNK_RES):
    """The round bounds R_1, R_2, ... of DESIGN.md section 14, given each selected protein's length and L: a protein
    stays active after R_g while one of its columns has L > R_g."""
    k = len(scored.dtype.names)
    wcap = max(chunk_res // 32, k) // k * 32
    last = np.max(np.stack([scored[n] for n in scored.dtype.names]), axis=0)
    out, r, active = [], 0, np.ones(len(lens), dtype=bool)
    while active.any() and r < K:
        res = max(int(lens[active].sum()), 1)
        wmin = -(-chunk_res // res)
        w = min(K - r, max(r if r else (K if h > K // 4 else max(64, 4 * h)), wmin))
        if K - r - w < wmin:
            w = K - r
        r += min(w, wcap)
        out.append(r)
        active &= last > r
    return out


def assert_rows(got, want, what):
    for n in want.dtype.names:
        bad = np.nonzero(got[n] != want[n])[0]
        assert len(bad) == 0, f"{what}, {n}: {len(bad)} rows differ, first {bad[:10].tolist()}"


# ---------------------------------------------------------------------------------------------- CPU
def test_seq_pvalues_formula():
    h, K = 3, 100
    dt = [(n, "<i8") for n in ("llr", "core_score", "has_core")]
    counts = np.array([(3, 0, 1), (3, 2, 3), (1, 3, 0)], dtype=dt)
    scored = np.array([(5, 100, 100), (100, 100, 7), (100, 40, 100)], dtype=dt)
    p = plaac_b200.seq_pvalues(counts, scored, h, K)
    assert p.dtype.names == ("llr", "core_score")
    assert p["llr"].tolist() == [3 / 5, 3 / 100, 2 / 101]  # (count == h at L == K_max: h / K_max)
    assert p["core_score"].tolist() == [1 / 101, 3 / 101, 3 / 40]
    # K_max == 0: nothing scored, p = 1
    z = np.zeros(2, dtype=dt)
    assert plaac_b200.seq_pvalues(z, z, 1, 0)["llr"].tolist() == [1.0, 1.0]


def test_bad_arguments_raise_before_the_call():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQN")])
    for kw, what in ((dict(columns=("core_score", "nosuch")), "null columns"), (dict(stop_hits=0), "stop_hits"),
                     (dict(stop_hits=-1), "stop_hits"), (dict(max_replicates=-1), "max_replicates")):
        a = dict(max_replicates=5)
        a.update(kw)
        with pytest.raises(ValueError, match=what):
            plaac_b200.Scorer.shuffle_null_seq(None, codes, offs, **a)  # (no ctx is needed to reject them)


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
    (["--stop-hits", "5"], "--stop-hits needs --null"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "0"], "--stop-hits needs H >= 1"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "-2"], "--stop-hits needs H >= 1"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "2.5"], "--stop-hits needs an integer"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "x"], "--stop-hits needs an integer"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", ""], "--stop-hits needs an integer"),
    # the checks of --null come first, as without --stop-hits
    (["--null", "NF", "--stop-hits", "3"], "--replicates"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "3", "-p", "all"], "cannot be combined with -p"),
    (["--null", "NF", "--replicates", "5", "--stop-hits", "3", "--null-columns", "Nope"], "unknown column 'Nope'"),
])
def test_cli_stop_hits_rejections(cli, tmp_path, args, why):
    fa = tmp_path / "s.fa"
    fa.write_text(">a\nMQQNPSD\n")
    nf = tmp_path / "null.txt"
    r = run(cli, "-s", "-i", str(fa), *[str(nf) if a == "NF" else a for a in args])
    assert r.returncode == 2 and why in r.stderr, r.stderr
    assert r.stdout == "" and not nf.exists()


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def scorer():
    s = plaac_b200.Scorer()
    yield s
    s.close()


SEED = 4321


@pytest.fixture(scope="module")
def fixed(scorer, golden):
    """The batch and the fixed call's values at K = 1000 (the first K replicates of each protein for every smaller K)."""
    codes, offs = null_batch(golden)
    counts, vals, obs = scorer.shuffle_null(codes, offs, 1000, seed=SEED, columns=NAMES, values=True, observed=True)
    return codes, offs, vals, obs


@pytest.mark.gpu
def test_exact_against_the_definition(scorer, fixed):
    codes, offs, vals, obs = fixed
    lens = np.diff(offs)
    first = later = never = edge = 0
    small = plaac_b200.Scorer()
    small.set_chunk(SMALL, 0)
    try:
        for sc, chunk_res in ((scorer, CHUNK_RES), (small, SMALL)):
            for K in (1, 37, 1000):
                for h in (1, 3, 10):
                    c, L, o = sc.shuffle_null_seq(codes, offs, K, stop_hits=h, seed=SEED, columns=NAMES, observed=True)
                    what = f"h = {h}, K_max = {K}, chunk bound {chunk_res}"
                    assert o.tobytes() == obs.tobytes(), what
                    wc, wl = restate(vals, obs, NAMES, h, K)
                    assert_rows(c, wc, "counts, " + what)
                    assert_rows(L, wl, "scored, " + what)
                    R = bounds(lens, L, h, K, chunk_res)
                    for n in NAMES:
                        stop = c[n] == h
                        first += int((stop & (L[n] <= R[0])).sum())
                        later += int((stop & (L[n] > R[0])).sum())
                        never += int((~stop).sum())
                        edge += int((stop & np.isin(L[n], R)).sum())  # on the last replicate of a round
    finally:
        small.close()
    assert first and later and never and edge, (first, later, never, edge)
    assert np.isnan(obs["core_score"]).any() and np.isneginf(obs["llr"]).any()
    # the default columns, in NULL_COLUMNS order
    c, L = scorer.shuffle_null_seq(codes, offs, 1000, seed=SEED)
    assert c.dtype.names == ("llr", "core_score", "hmm_all") and L.dtype == c.dtype
    wc, wl = restate(vals, obs, DEFAULT, 10, 1000)
    assert_rows(c, wc, "default columns")
    assert_rows(L, wl, "default columns")
    p = plaac_b200.seq_pvalues(c, L, 10, 1000)
    assert (p["llr"] > 0).all() and (p["llr"] <= 1).all()


@pytest.mark.gpu
def test_more_stop_hits_than_replicates_is_the_fixed_call(scorer, fixed):
    codes, offs, vals, obs = fixed
    for K in (37, 1000):
        c, L, o = scorer.shuffle_null_seq(codes, offs, K, stop_hits=K + 1, seed=SEED, columns=NAMES, observed=True)
        want = scorer.shuffle_null(codes, offs, K, seed=SEED, columns=NAMES)
        assert_rows(c, want, f"K = {K}")
        assert all((L[n] == K).all() for n in NAMES)
        assert o.tobytes() == scorer.score(codes, offs).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("how", ["chunked", "flag_budget", "long_fixed", "long_off", "long_auto", "kernel_variant_1",
                                 "generic_windows", "pinned", "subset"])
def test_invariance(fixed, how):
    codes, offs, vals, obs = fixed
    h, K = 3, 1000
    params = plaac_b200.default_params(ww1=31, ww2=41) if how == "generic_windows" else None
    sc = plaac_b200.Scorer(params)
    nprot = len(offs) - 1
    want_c, want_l = restate(vals, obs, NAMES, h, K)
    try:
        # (a small chunk bound, so that the proteins' runs take several rounds)
        if how == "chunked":
            sc.set_chunk(SMALL, 300)  # many chunks that cut proteins' replicate runs
        elif how == "flag_budget":
            sc.set_chunk(1 << 16, 300)  # a 2048-word flag budget: the longer rounds run as several sub-rounds
        else:
            sc.set_chunk(SMALL, 0)
        if how == "kernel_variant_1":
            sc.set_kernel_variant(1)
        elif how.startswith("long_"):
            sc.set_long_path({"long_fixed": 1024, "long_off": 0, "long_auto": -1}[how])
        if how == "subset":
            sel = np.array([5, 0, nprot - 1, 5, 17, 2, nprot - 3, 0], dtype=np.int32)
            c, L, o = sc.shuffle_null_seq(codes, offs, K, stop_hits=h, seed=SEED, columns=NAMES, proteins=sel, observed=True)
            assert_rows(c, want_c[sel], how)
            assert_rows(L, want_l[sel], how)
            assert o.tobytes() == obs[sel].tobytes()
            return
        if how == "pinned":
            nl = plaac_b200.Null(replicates=K, seed=SEED, columns=ALL, reserved=0, nsel=-1, proteins=None)
            with plaac_b200.PinnedBuffer(nprot, dtype=want_c.dtype) as cb, \
                    plaac_b200.PinnedBuffer(nprot, dtype=want_c.dtype) as lb, \
                    plaac_b200.PinnedBuffer(nprot, dtype=plaac_b200.SUMMARY_DTYPE) as ob:
                nl.counts = cb.array.ctypes.data
                rc = plaac_b200.lib().plaac_score_shuffles_seq(sc._h, codes.ctypes.data, offs.ctypes.data, nprot, C.byref(nl),
                                                               h, lb.array.ctypes.data, ob.array.ctypes.data)
                assert rc == 0
                c, L, o = cb.array.copy(), lb.array.copy(), ob.array.copy()
            assert o.tobytes() == obs.tobytes()
        else:
            c, L = sc.shuffle_null_seq(codes, offs, K, stop_hits=h, seed=SEED, columns=NAMES)
        if how in ("generic_windows", "kernel_variant_1"):
            # records of their own: compare with the fixed call of the same ctx
            _, v2, o2 = sc.shuffle_null(codes, offs, K, seed=SEED, columns=NAMES, values=True, observed=True)
            want_c, want_l = restate(v2, o2, NAMES, h, K)
    finally:
        sc.close()
    assert_rows(c, want_c, how)
    assert_rows(L, want_l, how)


@pytest.mark.gpu
def test_long_protein_stops_in_a_late_round():
    codes, offs = synth.long_proteins(seed=47, lengths=(34000,))
    K, seed = 2000, 77
    scorer = plaac_b200.Scorer()
    scorer.set_chunk(SMALL, 0)  # rounds of 64, 64, 128, ... replicates instead of one of 2 000
    _, vals, obs = scorer.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, values=True, observed=True)
    # h and a column that stops after the first round: its h-th hit comes after R_1 (>= max(64, 4h))
    never = np.full(1, K, dtype=[("x", "<i8")])

    def R1(h):
        return bounds(np.diff(offs), never, h, K, SMALL)[0]

    pick = [(h, n) for h in range(1, 40) for n in NAMES
            if hits_of(vals, obs, n)[0].sum() >= h and np.argmax(np.cumsum(hits_of(vals, obs, n)[0]) >= h) + 1 > R1(h)]
    assert pick
    h, late = pick[0]
    want_c, want_l = restate(vals, obs, NAMES, h, K)
    assert want_c[late][0] == h and want_l[late][0] > R1(h)
    for thr in (-1, 1024):
        scorer.set_long_path(thr)
        try:
            c, L = scorer.shuffle_null_seq(codes, offs, K, stop_hits=h, seed=seed, columns=NAMES)
        finally:
            scorer.set_long_path(-1)
        assert_rows(c, want_c, f"threshold {thr}")
        assert_rows(L, want_l, f"threshold {thr}")
    assert len(bounds(np.diff(offs), want_l, h, K, SMALL)) >= 2
    scorer.close()


@pytest.mark.gpu
def test_flag_budget_exceeded(golden):
    """20 000 copies of Sup35p, every row active into the round [1024, 2048): 6.1e7 flag bits, over a budget of 1.7e7
    (one bit per residue of a 2^24-residue chunk bound), so that round runs as 4 sub-rounds."""
    codes, offs = plaac_b200.pack([plaac_b200.encode(p["seq"]) for p in golden["proteins"] if p["name"] == "Sup35p"])
    K, h, n = 2048, 10, 20000
    sc = plaac_b200.Scorer()
    try:
        _, vals, obs = sc.shuffle_null(codes, offs, K, seed=SEED, values=True, observed=True)
        want_c, want_l = restate(vals, obs, DEFAULT, h, K)
        assert max(int(want_l[c][0]) for c in DEFAULT) > 1024  # (the round over budget is reached)
        sc.set_chunk(1 << 24, 0)
        c, L = sc.shuffle_null_seq(codes, offs, K, stop_hits=h, seed=SEED, proteins=np.zeros(n, dtype=np.int32))
    finally:
        sc.close()
    for f in DEFAULT:
        assert (c[f] == want_c[f][0]).all() and (L[f] == want_l[f][0]).all(), f


def _call(sc, codes, offs, nprot, K, h, nsel, proteins, counts, scored, values=None, observed=None, reserved=0, seed=0):
    nl = plaac_b200.Null(replicates=K, seed=seed, columns=ALL, reserved=reserved, nsel=nsel, proteins=proteins,
                         counts=counts, values=values)
    rc = plaac_b200.lib().plaac_score_shuffles_seq(sc._h, codes, offs, nprot, C.byref(nl), h, scored, observed)
    return rc, plaac_b200.lib().plaac_last_error(sc._h).decode()


@pytest.mark.gpu
def test_errors_and_edges(scorer):
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDQQNKLLAPQ"), plaac_b200.encode("ACDEFG")])
    cp, op = codes.ctypes.data, offs.ctypes.data
    sel = np.array([1, 0], dtype=np.int32)
    cnt = np.full(2 * 14, 7, dtype=np.int64)
    sco = np.full(2 * 14, 7, dtype=np.int64)
    vals = np.zeros(2 * 4 * 14)
    base = dict(K=4, h=2, nsel=2, proteins=sel.ctypes.data, counts=cnt.ctypes.data, scored=sco.ctypes.data)
    for kw, what in [(dict(h=0), "stop_hits 0"), (dict(h=-1), "stop_hits -1"), (dict(values=vals.ctypes.data), "values"),
                     (dict(scored=None), "NULL scored"), (dict(nsel=-1, scored=None), "NULL scored"),
                     (dict(reserved=1), "reserved"), (dict(K=-1), "replicates -1"), (dict(counts=None), "NULL counts")]:
        a = dict(base)
        a.update(kw)
        rc, msg = _call(scorer, cp, op, 2, a["K"], a["h"], a["nsel"], a["proteins"], a["counts"], a["scored"],
                        values=a.get("values"), reserved=a.get("reserved", 0))
        assert rc == -1 and what in msg and msg.startswith("plaac_score_shuffles_seq"), (kw, msg)
    for bad in ([0, 2], [-1, 0]):
        b = np.array(bad, dtype=np.int32)
        j = next(k for k, x in enumerate(bad) if not 0 <= x < 2)
        rc, msg = _call(scorer, cp, op, 2, 4, 2, len(b), b.ctypes.data, cnt.ctypes.data, sco.ctypes.data)
        assert rc == -1 and f"selected protein {j}: index {bad[j]}" in msg, msg
    # K_max == 0: counts and scored are 0, observed is written
    obs = np.zeros(2, dtype=plaac_b200.SUMMARY_DTYPE)
    rc, _ = _call(scorer, cp, op, 2, 0, 2, 2, sel.ctypes.data, cnt.ctypes.data, sco.ctypes.data, observed=obs.ctypes.data)
    assert rc == 0 and (cnt == 0).all() and (sco == 0).all()
    assert obs.tobytes() == scorer.score(codes, offs)[sel].tobytes()
    # nsel == 0: PLAAC_OK, nothing written
    cnt[:] = 7
    rc, _ = _call(scorer, cp, op, 2, 4, 2, 0, sel.ctypes.data, None, None)
    assert rc == 0 and (cnt == 7).all()
    c, L = scorer.shuffle_null_seq(codes, offs, 3, proteins=[])
    assert len(c) == 0 and len(L) == 0


@pytest.mark.gpu
def test_invalid_reference_bytes_everything_written(scorer):
    codes, offs = reference_batch()
    codes = codes.copy()
    codes[offs[3] + 1] = 30
    codes[offs[50] + 7] = 200
    nprot = len(offs) - 1
    K, h, seed = 300, 3, 3
    sel = np.array([3, 50, 7, 3], dtype=np.int32)
    counts = np.full(len(sel), -1, dtype=[(n, "<i8") for n in NAMES])
    scored = np.full(len(sel), -1, dtype=counts.dtype)
    obs = np.zeros(len(sel), dtype=plaac_b200.SUMMARY_DTYPE)
    rc, msg = _call(scorer, codes.ctypes.data, offs.ctypes.data, nprot, K, h, len(sel), sel.ctypes.data,
                    counts.ctypes.data, scored.ctypes.data, observed=obs.ctypes.data, seed=seed)
    assert rc == -1 and "> 21" in msg, msg
    vals = np.zeros((len(sel), K), dtype=[(n, "<f8") for n in NAMES])
    fc = np.zeros(len(sel), dtype=counts.dtype)
    fo = np.zeros(len(sel), dtype=plaac_b200.SUMMARY_DTYPE)
    nl = plaac_b200.Null(replicates=K, seed=seed, columns=ALL, reserved=0, nsel=len(sel), proteins=sel.ctypes.data,
                         counts=fc.ctypes.data, values=vals.ctypes.data)
    assert plaac_b200.lib().plaac_score_shuffles(scorer._h, codes.ctypes.data, offs.ctypes.data, nprot, C.byref(nl),
                                                 fo.ctypes.data) == -1
    assert obs.tobytes() == fo.tobytes()
    want_c, want_l = restate(vals, fo, NAMES, h, K)
    assert_rows(counts, want_c, "counts with bytes > 21")
    assert_rows(scored, want_l, "scored with bytes > 21")


@pytest.mark.gpu
def test_cli_null_file_matches_the_api(cli, scorer, tmp_path, golden):
    names = [p["name"] for p in golden["proteins"]] + ["short"]
    seqs = [p["seq"].rstrip("*") for p in golden["proteins"]] + ["QNQ"]
    fa = tmp_path / "small.fa"
    fa.write_text(_fasta(names, seqs))
    codes, offs = plaac_b200.pack([plaac_b200.encode(s) for s in seqs])
    K, h = 500, 5
    plain = run(cli, "-s", "-i", str(fa))
    assert plain.returncode == 0, plain.stderr
    for cols, arg in ((DEFAULT, []), (("llr", "papa_combo", "has_core"), ["--null-columns", "hasCORE,PAPAcombo,LLR"])):
        nf = tmp_path / "null.txt"
        r = run(cli, "-s", "-i", str(fa), "--null", str(nf), "--replicates", str(K), "--stop-hits", str(h), *arg)
        assert r.returncode == 0, r.stderr
        assert r.stdout == plain.stdout
        lines = nf.read_text().rstrip("\n").split("\n")
        head = ["SEQid"]
        for n in cols:
            cn = CLI_NAMES[NAMES.index(n)]
            head += [f"r{cn}", f"n{cn}"] + ([] if n == "has_core" else [f"p{cn}"])
        assert lines[0].split("\t") == head
        printed = [x.split("\t")[0] for x in plain.stdout.rstrip("\n").split("\n")[1:]]
        assert [x.split("\t")[0] for x in lines[1:]] == printed
        c, L = scorer.shuffle_null_seq(codes, offs, K, stop_hits=h, columns=cols)
        p = plaac_b200.seq_pvalues(c, L, h, K)
        row = {nm: i for i, nm in enumerate(names)}
        for line in lines[1:]:
            cells = line.split("\t")
            j = row[cells[0]]
            exp = []
            for n in cols:
                exp += [str(int(L[n][j])), str(int(c[n][j]))] + ([] if n == "has_core" else ["%.6g" % p[n][j]])
            assert cells[1:] == exp, (line, exp)
