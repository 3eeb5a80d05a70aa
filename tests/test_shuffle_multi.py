"""Shuffle nulls on several ctxs (plaac_score_shuffles_multi, plaac_score_shuffles_seq_multi, MultiScorer.shuffle_null
and MultiScorer.shuffle_null_seq; DESIGN.md section 15).  Every result is compared byte for byte with the single call on
one Scorer.  With two GPUs the ctxs go to devices [0, 1] and [0, 1, 0], otherwise all to device 0."""
import ctypes as C

import numpy as np
import pytest

import plaac_b200
from tests import synth
from tests.test_shuffle_null import ALL, NAMES, null_batch
from tests.test_variants import reference_batch

SEED = 4321
SMALL = 1 << 20  # a chunk bound that makes the sequential rounds short: many rounds


def devices(nctx):
    two = plaac_b200.lib().plaac_device_count() >= 2
    return [k % 2 if two else 0 for k in range(nctx)]


def part_starts(W, nctx):
    return [W * c // nctx for c in range(nctx + 1)]


def same(got, want, what):
    got, want = (got, want) if isinstance(want, tuple) else ((got,), (want,))
    assert len(got) == len(want), what
    for k, (g, w) in enumerate(zip(got, want)):
        assert g.dtype == w.dtype and g.shape == w.shape, (what, k)
        assert g.tobytes() == w.tobytes(), (what, k)


# ---------------------------------------------------------------------------------------------- CPU
def test_bad_arguments_raise_before_the_call():
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQN")])
    for cols in (("core_score", "nosuch"), (), ("mw_score",)):
        with pytest.raises(ValueError, match="null columns"):
            plaac_b200.MultiScorer.shuffle_null(None, codes, offs, 5, columns=cols)  # (no ctx is needed to reject them)
        with pytest.raises(ValueError, match="null columns"):
            plaac_b200.MultiScorer.shuffle_null_seq(None, codes, offs, 5, columns=cols)
    for kw, what in ((dict(stop_hits=0), "stop_hits"), (dict(max_replicates=-1), "max_replicates")):
        a = dict(max_replicates=5)
        a.update(kw)
        with pytest.raises(ValueError, match=what):
            plaac_b200.MultiScorer.shuffle_null_seq(None, codes, offs, **a)


def test_part_starts_cover_the_span():
    for W in (0, 1, 2, 5, 257, 10**6):
        for n in (1, 2, 3, 8):
            p = part_starts(W, n)
            assert p[0] == 0 and p[-1] == W and all(b - a in (W // n, W // n + 1) for a, b in zip(p, p[1:]))


# ---------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def single():
    s = plaac_b200.Scorer()
    yield s
    s.close()


@pytest.fixture(scope="module")
def multis():
    ms = {n: plaac_b200.MultiScorer(devices=devices(n)) for n in (2, 3)}
    yield ms
    for m in ms.values():
        m.close()


@pytest.fixture(scope="module")
def batch(golden):
    return null_batch(golden)


def selection(offs):
    nprot = len(offs) - 1
    return np.array([5, 0, nprot - 1, 5, 17, 2, nprot - 3, 0], dtype=np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("nctx", [2, 3])
def test_fixed_call_equals_the_single_call(single, multis, batch, nctx):
    codes, offs = batch
    ms = multis[nctx]
    for K in (0, 1, 2, 257):  # (K = 2 with 3 ctxs: one ctx scores nothing)
        for sel in (None, selection(offs)):
            what = f"nctx = {nctx}, K = {K}, selection {sel is not None}"
            kw = dict(seed=SEED, columns=NAMES, proteins=sel)
            want = single.shuffle_null(codes, offs, K, values=True, observed=True, **kw)
            same(ms.shuffle_null(codes, offs, K, values=True, observed=True, **kw), want, what)
            same(ms.shuffle_null(codes, offs, K, **kw), want[0], what + ", counts only")
    same(ms.shuffle_null(codes, offs, 100, seed=7), single.shuffle_null(codes, offs, 100, seed=7), "default columns")


@pytest.mark.gpu
@pytest.mark.parametrize("nctx", [2, 3])
def test_fixed_call_one_long_protein(single, multis, nctx):
    codes, offs = synth.long_proteins(seed=47, lengths=(34000,))
    kw = dict(seed=77, columns=NAMES, values=True, observed=True)
    same(multis[nctx].shuffle_null(codes, offs, 64, **kw), single.shuffle_null(codes, offs, 64, **kw), f"nctx = {nctx}")


@pytest.mark.gpu
@pytest.mark.parametrize("nctx", [2, 3])
def test_sequential_call_equals_the_single_call(single, multis, batch, nctx):
    codes, offs = batch
    ms = multis[nctx]
    stopped = 0
    for seed in (SEED, 99):
        for K in (1, 37, 1000):
            for h in (1, 3, 10, K + 1):
                for sel in (None, selection(offs)):
                    what = f"nctx = {nctx}, seed {seed}, K_max = {K}, h = {h}, selection {sel is not None}"
                    kw = dict(stop_hits=h, seed=seed, columns=NAMES, proteins=sel, observed=True)
                    want = single.shuffle_null_seq(codes, offs, K, **kw)
                    got = ms.shuffle_null_seq(codes, offs, K, **kw)
                    same(got, want, what)
                    stopped += sum(int((want[0][n] == h).sum()) for n in NAMES)
                    if h > K:  # nothing stops: the fixed call's counts, L = K_max
                        same(got[0], single.shuffle_null(codes, offs, K, seed=seed, columns=NAMES, proteins=sel), what)
                        assert all((got[1][n] == K).all() for n in NAMES), what
    assert stopped > 0
    same(ms.shuffle_null_seq(codes, offs, 500), single.shuffle_null_seq(codes, offs, 500), "default columns")


@pytest.mark.gpu
@pytest.mark.parametrize("nctx", [2, 3])
def test_single_round_stops_in_every_part(single, multis, batch, nctx):
    """h > K_max / 4: the schedule runs one round over [0, K_max), cut into the parts floor(K_max c / nctx); some column
    stops in each part, so every ctx's stops are found and merged, not only the first ctx's."""
    codes, offs = batch
    K, h = 300, 80
    kw = dict(stop_hits=h, seed=SEED, columns=NAMES, observed=True)
    want = single.shuffle_null_seq(codes, offs, K, **kw)
    same(multis[nctx].shuffle_null_seq(codes, offs, K, **kw), want, f"nctx = {nctx}")
    p = part_starts(K, nctx)
    c, L = want[0], want[1]
    for k in range(nctx):
        n_in = sum(int(((c[n] == h) & (L[n] > p[k]) & (L[n] <= p[k + 1])).sum()) for n in NAMES)
        assert n_in > 0, (k, p)


@pytest.mark.gpu
@pytest.mark.parametrize("nctx", [2, 3])
def test_sequential_call_one_long_protein(single, nctx):
    """A 34 000-residue protein: columns that stop (in a later round, with a small chunk bound) and columns that never do."""
    codes, offs = synth.long_proteins(seed=47, lengths=(34000,))
    K = 2000
    ms = plaac_b200.MultiScorer(devices=devices(nctx))
    try:
        for s in ms.scorers:
            s.set_chunk(SMALL, 0)
        stops = runs = 0
        for h in (1, 3, 10, 40):
            kw = dict(stop_hits=h, seed=77, columns=NAMES, observed=True)
            want = single.shuffle_null_seq(codes, offs, K, **kw)
            same(ms.shuffle_null_seq(codes, offs, K, **kw), want, f"nctx = {nctx}, h = {h}")
            stops += sum(int(want[0][n][0] == h and want[1][n][0] > 64) for n in NAMES)
            runs += sum(int(want[0][n][0] < h) for n in NAMES)
    finally:
        ms.close()
    assert stops > 0 and runs > 0, (stops, runs)


# the columns every kernel variant computes to the same bytes (variant 1 has PAPA columns of its own)
VARIANT_SAFE = ("llr", "core_score", "prd_score", "hmm_all", "hmm_vit", "fi_meanhydro", "fi_meancharge", "fi_meancombo",
                "has_core")


@pytest.mark.gpu
def test_settings_that_differ_per_ctx(single, batch):
    """A small flag budget on one ctx only (global sub-rounds on all of them), the long path off on another, kernel
    variant 1 on a third."""
    codes, offs = batch
    ms = plaac_b200.MultiScorer(devices=devices(3))
    try:
        ms.scorers[0].set_long_path(0)
        ms.scorers[1].set_chunk(1 << 16, 300)  # a 2 048-word flag budget
        ms.scorers[2].set_kernel_variant(1)
        for K, h in ((1000, 3), (1000, 10), (400, 120)):
            kw = dict(stop_hits=h, seed=SEED, columns=VARIANT_SAFE, observed=True)
            want = single.shuffle_null_seq(codes, offs, K, **kw)
            same(ms.shuffle_null_seq(codes, offs, K, **kw), want, f"sequential, K_max = {K}, h = {h}")
        kw = dict(seed=SEED, columns=VARIANT_SAFE, values=True, observed=True)
        same(ms.shuffle_null(codes, offs, 300, **kw), single.shuffle_null(codes, offs, 300, **kw), "fixed")
    finally:
        ms.close()


def handles(ms):
    return (C.c_void_p * len(ms.scorers))(*[s._h for s in ms.scorers])


def raw_fixed(hs, nctx, codes, offs, nprot, K, nsel, proteins, counts, values=None, observed=None, columns=ALL, reserved=0,
              seed=0, spec=True):
    nl = plaac_b200.Null(replicates=K, seed=seed, columns=columns, reserved=reserved, nsel=nsel, proteins=proteins,
                         counts=counts, values=values)
    return plaac_b200.lib().plaac_score_shuffles_multi(hs, nctx, codes, offs, nprot, C.byref(nl) if spec else None, observed)


def raw_seq(hs, nctx, codes, offs, nprot, K, h, nsel, proteins, counts, scored, values=None, observed=None, columns=ALL,
            reserved=0, seed=0, spec=True):
    nl = plaac_b200.Null(replicates=K, seed=seed, columns=columns, reserved=reserved, nsel=nsel, proteins=proteins,
                         counts=counts, values=values)
    return plaac_b200.lib().plaac_score_shuffles_seq_multi(hs, nctx, codes, offs, nprot, C.byref(nl) if spec else None, h,
                                                           scored, observed)


def err(h):
    return plaac_b200.lib().plaac_last_error(h).decode()


@pytest.mark.gpu
def test_invalid_reference_bytes_as_the_single_call(single, multis):
    codes, offs = reference_batch()
    codes = codes.copy()
    codes[offs[3] + 1] = 30
    codes[offs[50] + 7] = 200
    nprot = len(offs) - 1
    sel = np.array([3, 50, 7, 3], dtype=np.int32)
    K, h, seed = 300, 3, 3
    cdt = [(n, "<i8") for n in NAMES]

    def fixed(hs, nctx):
        counts = np.full(len(sel), -1, dtype=cdt)
        vals = np.full((len(sel), K), np.inf, dtype=[(n, "<f8") for n in NAMES])
        obs = np.zeros(len(sel), dtype=plaac_b200.SUMMARY_DTYPE)
        rc = raw_fixed(hs, nctx, codes.ctypes.data, offs.ctypes.data, nprot, K, len(sel), sel.ctypes.data,
                       counts.ctypes.data, vals.ctypes.data, obs.ctypes.data, seed=seed)
        return rc, err(hs[0]), counts, vals, obs

    def seq(hs, nctx):
        counts = np.full(len(sel), -1, dtype=cdt)
        scored = np.full(len(sel), -1, dtype=cdt)
        obs = np.zeros(len(sel), dtype=plaac_b200.SUMMARY_DTYPE)
        rc = raw_seq(hs, nctx, codes.ctypes.data, offs.ctypes.data, nprot, K, h, len(sel), sel.ctypes.data,
                     counts.ctypes.data, scored.ctypes.data, None, obs.ctypes.data, seed=seed)
        return rc, err(hs[0]), counts, scored, obs

    one = (C.c_void_p * 1)(single._h)
    want_f, want_s = fixed(one, 1), seq(one, 1)
    assert want_f[0] == want_s[0] == -1 and "> 21" in want_f[1] and "> 21" in want_s[1]
    for nctx, ms in multis.items():
        hs = handles(ms)
        for got, want in ((fixed(hs, nctx), want_f), (seq(hs, nctx), want_s)):
            assert got[:2] == want[:2], nctx
            for g, w in zip(got[2:], want[2:]):
                assert g.tobytes() == w.tobytes(), nctx


@pytest.mark.gpu
def test_errors(single, multis):
    codes, offs = plaac_b200.pack([plaac_b200.encode("MQQNPSDQQNKLLAPQ"), plaac_b200.encode("ACDEFG")])
    cp, op = codes.ctypes.data, offs.ctypes.data
    sel = np.array([1, 0], dtype=np.int32)
    cnt = np.full(2 * 14, 7, dtype=np.int64)
    sco = np.full(2 * 14, 7, dtype=np.int64)
    vals = np.zeros(2 * 4 * 14)
    ms = multis[2]
    hs = handles(ms)
    # the ctx list (the text is the global one: there is no ctx to hold it)
    for fn, call in (("plaac_score_shuffles_multi", lambda h, n: raw_fixed(h, n, cp, op, 2, 4, 2, sel.ctypes.data, cnt.ctypes.data)),
                     ("plaac_score_shuffles_seq_multi",
                      lambda h, n: raw_seq(h, n, cp, op, 2, 4, 2, 2, sel.ctypes.data, cnt.ctypes.data, sco.ctypes.data))):
        for h, n, what in ((hs, 0, "no contexts"), (hs, -1, "no contexts"), (None, 2, "no contexts"),
                           ((C.c_void_p * 2)(ms.scorers[0]._h, None), 2, "NULL ctx 1"),
                           ((C.c_void_p * 3)(None, ms.scorers[0]._h, ms.scorers[1]._h), 3, "NULL ctx 0")):
            assert call(h, n) == -1 and err(None) == f"{fn}: {what}", (fn, what, err(None))
    # every check of the single calls, with the multi call's name, on ctxs[0]
    fixed_cases = [(dict(K=-1), "replicates -1"), (dict(nsel=-2), "nsel -2"), (dict(reserved=1), "reserved"),
                   (dict(columns=0), "columns"), (dict(columns=1 << 14), "columns"), (dict(columns=-1), "columns"),
                   (dict(proteins=None), "NULL proteins"), (dict(counts=None), "NULL counts"),
                   (dict(nsel=-1, counts=None), "NULL counts"), (dict(spec=False), "NULL null_spec")]
    for kw, what in fixed_cases:
        a = dict(K=4, nsel=2, proteins=sel.ctypes.data, counts=cnt.ctypes.data)
        a.update(kw)
        args = (cp, op, 2, a.pop("K"), a.pop("nsel"), a.pop("proteins"), a.pop("counts"))
        rc1 = raw_fixed((C.c_void_p * 1)(single._h), 1, *args, **a)
        m1 = err(single._h)
        rc = raw_fixed(hs, 2, *args, **a)
        m = err(hs[0])
        assert rc == rc1 == -1 and what in m and m == m1.replace("plaac_score_shuffles", "plaac_score_shuffles_multi", 1), (kw, m, m1)
    seq_cases = [(dict(h=0), "stop_hits 0"), (dict(h=-1), "stop_hits -1"), (dict(values=vals.ctypes.data), "values"),
                 (dict(scored=None), "NULL scored"), (dict(nsel=-1, scored=None), "NULL scored"),
                 (dict(reserved=1), "reserved"), (dict(K=-1), "replicates -1"), (dict(counts=None), "NULL counts"),
                 (dict(columns=0), "columns"), (dict(nsel=-2), "nsel -2"), (dict(proteins=None), "NULL proteins"),
                 (dict(spec=False), "NULL null_spec")]
    for kw, what in seq_cases:
        a = dict(K=4, h=2, nsel=2, proteins=sel.ctypes.data, counts=cnt.ctypes.data, scored=sco.ctypes.data)
        a.update(kw)
        args = (cp, op, 2, a.pop("K"), a.pop("h"), a.pop("nsel"), a.pop("proteins"), a.pop("counts"), a.pop("scored"))
        rc1 = raw_seq((C.c_void_p * 1)(single._h), 1, *args, **a)
        m1 = err(single._h)
        rc = raw_seq(hs, 2, *args, **a)
        m = err(hs[0])
        assert rc == rc1 == -1 and what in m and m == m1.replace("plaac_score_shuffles_seq", "plaac_score_shuffles_seq_multi", 1), (kw, m, m1)
    for bad in ([0, 2], [-1, 0], [1, 1, 0, 5]):
        b = np.array(bad, dtype=np.int32)
        j = next(k for k, x in enumerate(bad) if not 0 <= x < 2)
        assert raw_fixed(hs, 2, cp, op, 2, 4, len(b), b.ctypes.data, cnt.ctypes.data) == -1
        assert err(hs[0]).startswith("plaac_score_shuffles_multi: ") and f"selected protein {j}: index {bad[j]}" in err(hs[0])
        assert raw_seq(hs, 2, cp, op, 2, 4, 2, len(b), b.ctypes.data, cnt.ctypes.data, sco.ctypes.data) == -1
        assert err(hs[0]).startswith("plaac_score_shuffles_seq_multi: ") and f"selected protein {j}: index {bad[j]}" in err(hs[0])
    # nsel == 0 and K == 0, as the single calls
    cnt[:] = 7
    assert raw_fixed(hs, 2, cp, op, 2, 4, 0, sel.ctypes.data, None) == 0 and (cnt == 7).all()
    assert raw_seq(hs, 2, cp, op, 2, 4, 2, 0, sel.ctypes.data, None, None) == 0
    obs = np.zeros(2, dtype=plaac_b200.SUMMARY_DTYPE)
    assert raw_seq(hs, 2, cp, op, 2, 0, 2, 2, sel.ctypes.data, cnt.ctypes.data, sco.ctypes.data, observed=obs.ctypes.data) == 0
    assert (cnt == 0).all() and (sco == 0).all() and obs.tobytes() == single.score(codes, offs)[sel].tobytes()
    assert len(ms.shuffle_null(codes, offs, 3, proteins=[])) == 0
    c, L = ms.shuffle_null_seq(codes, offs, 3, proteins=[])
    assert len(c) == 0 and len(L) == 0


@pytest.mark.gpu
def test_distinct_devices_yeast_sized():
    """Every GPU of the box, each its own device, on a yeast-sized synthetic set; skipped on a one-GPU box, where the
    other tests put every ctx on device 0."""
    ndev = plaac_b200.lib().plaac_device_count()
    if ndev < 2:
        pytest.skip("needs >= 2 GPUs (plaac_device_count() = %d)" % ndev)
    codes, offs = synth.proteome(6000, seed=48)
    one = plaac_b200.Scorer(device=0)
    ms = plaac_b200.MultiScorer(devices=list(range(ndev)))
    try:
        kw = dict(seed=5, observed=True)
        same(ms.shuffle_null(codes, offs, 200, **kw), one.shuffle_null(codes, offs, 200, **kw), "fixed")
        kw = dict(stop_hits=10, seed=5, observed=True)
        same(ms.shuffle_null_seq(codes, offs, 20000, **kw), one.shuffle_null_seq(codes, offs, 20000, **kw), "sequential")
    finally:
        ms.close()
        one.close()
