"""The throughput summary kernel tests FoldIndex runs and the PAPA gate in exact 32-bit integers where the host can prove
that this gives the FP64 signs (plan_int_fold).  Every byte must stay what variant 2 (FP64 running sums) produces:
at exact integer zeros (the kernel then scores the bucket again with FP64 sums), at window edges, for parameters that
fail the proof and at the widest windows."""
import numpy as np
import pytest

import plaac_b200
from tests import synth

pytestmark = pytest.mark.gpu


def _same_bytes(params, codes, offs):
    a = plaac_b200.Scorer(params)
    a.set_kernel_variant(2)
    b = plaac_b200.Scorer(params)
    ra, rb = a.score(codes, offs), b.score(codes, offs)
    a.close()
    b.close()
    assert ra.tobytes() == rb.tobytes()


def _papa_zero_proteins(nres=30_000_000, seed=5, w=20, flank=150):
    """Stretches centred where the PAPA gate's integer form 557 Th - 18000 Tac - 20718 W is exactly 0 (default tables:
    hydropathy h/90, W = (2w+1)^2), found by scanning a long random sequence."""
    P = plaac_b200.default_params()
    hyd = np.rint(np.ctypeslib.as_array(P.hydro2) * 90).astype(np.int64)
    chg = np.ctypeslib.as_array(P.charge).astype(np.int64)
    rng = np.random.default_rng(seed)
    # neutral residues and about 1 in 7 positively charged: window charge sums near 41/7, Tac near 228 and Th near the
    # 69894 that goes with it
    neutral = np.nonzero(chg[:21] == 0)[0]
    neutral = neutral[neutral > 0]
    plus = np.nonzero(chg[:21] > 0)[0]
    seq = neutral[rng.integers(0, len(neutral), nres)].astype(np.uint8)
    pick = rng.random(nres) < 0.136
    seq[pick] = plus[rng.integers(0, len(plus), int(pick.sum()))]
    full = 2 * w + 1
    tri = np.concatenate([np.arange(1, full + 1), np.arange(full - 1, 0, -1)])
    th = np.convolve(hyd[seq], tri, mode="valid")                                 # centres 2w .. nres-1-2w
    sl = np.abs(np.convolve(chg[seq], np.ones(full, np.int64), mode="valid"))    # centres w .. nres-1-w
    tac = np.convolve(sl, np.ones(full, np.int64), mode="valid")                  # centres 2w .. nres-1-2w
    v = 557 * th - 18000 * tac - 20718 * full * full
    hits = np.nonzero(v == 0)[0] + 2 * w
    hits = hits[(hits >= flank) & (hits < nres - flank)]
    return [seq[c - flank:c + flank + 1 + (i % 7)].copy() for i, c in enumerate(hits)]


def test_exact_zero_papa_gates():
    seqs = _papa_zero_proteins()
    assert len(seqs) >= 5
    codes, offs = plaac_b200.pack(seqs)
    _same_bytes(None, codes, offs)


def test_lengths_around_the_window_edges():
    rng = np.random.default_rng(11)
    for ww in (41, 40, 61, 13):
        w = ww // 2
        lens = sorted({max(1, x) for c in (w, 2 * w + 1, 4 * w, 4 * w + 2, (ww - 1) // 2) for x in range(c - 3, c + 4)})
        seqs = [rng.integers(0, 22, n).astype(np.uint8) for n in lens for _ in range(40)]
        codes, offs = plaac_b200.pack(seqs)
        _same_bytes(plaac_b200.default_params(ww1=ww, ww2=ww), codes, offs)


def test_parameters_that_fail_the_proof():
    codes, offs = synth.proteome(20_000, seed=81, median=290.0, sigma=0.62)
    P = plaac_b200.default_params()
    P.hydro2[5] = P.hydro2[5] + 1e-7          # no longer h/90
    _same_bytes(P, codes, offs)
    P = plaac_b200.default_params()
    P.fi_cc[0] = 2.785 + 3e-12                # no small denominator
    _same_bytes(P, codes, offs)


@pytest.mark.parametrize("ww", [61, 205, 255])
def test_wide_windows(ww):
    codes, offs = synth.proteome(6_000, seed=82, median=600.0, sigma=0.5)
    _same_bytes(plaac_b200.default_params(ww1=ww, ww2=ww), codes, offs)
