"""Host-side (numpy) synthetic proteomes for the parity tests, SURVEY.md section 8(d):
log-normal lengths, residues iid from a background, X at 1e-4, a Q/N-rich
segment drawn from the prion-domain composition injected into 5 % of proteins."""
import numpy as np

BG_SCER = np.array([0, 0.0550, 0.0126, 0.0586, 0.0655, 0.0441, 0.0498, 0.0217, 0.0655, 0.0735, 0.0950, 0.0207,
                    0.0615, 0.0438, 0.0396, 0.0444, 0.0899, 0.0592, 0.0556, 0.0104, 0.0337, 0])
PRD_28 = np.array([0, 0.04865, 0.00219, 0.01638, 0.00783, 0.02537, 0.07603, 0.0181, 0.02018, 0.01641, 0.02639,
                   0.02975, 0.25885, 0.05126, 0.15178, 0.025, 0.10988, 0.03841, 0.01972, 0.00157, 0.05624, 0])


def proteome(nprot, seed, median=407.0, sigma=0.66, min_len=16, max_len=40000, prd_rate=0.05, x_rate=1e-4,
             bg=BG_SCER):
    rng = np.random.default_rng(seed)
    lens = np.clip(np.rint(rng.lognormal(np.log(median), sigma, nprot)), min_len, max_len).astype(np.int64)
    offsets = np.zeros(nprot + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    ntot = int(offsets[-1])
    p = bg / bg.sum()
    codes = rng.choice(22, size=ntot, p=p).astype(np.uint8)
    codes[rng.random(ntot) < x_rate] = 0
    pp = PRD_28 / PRD_28.sum()
    for i in np.nonzero(rng.random(nprot) < prd_rate)[0]:
        n = int(lens[i])
        seg = int(min(n, rng.integers(60, 301)))
        st = int(rng.integers(0, n - seg + 1))
        codes[offsets[i] + st: offsets[i] + st + seg] = rng.choice(22, size=seg, p=pp)
    return codes, offsets


def repeat_proteome(nprot, seed):
    """Yeast-like proteins whose Q/N-rich parts repeat, as real prion domains do, so that several windows of the
    60-residue LLR and CORE searches have the same composition: in turn a block and a copy of it, a block and a
    permutation of it, and an oligopeptide repeat.  Which of such windows the reference picks is decided by the
    rounding of its running sums (over the -1e6 mask outside the PrD for the CORE)."""
    rng = np.random.default_rng(seed)
    bg, prd = BG_SCER / BG_SCER.sum(), PRD_28 / PRD_28.sum()
    seqs = []
    for i in range(nprot):
        n = int(np.clip(np.rint(rng.lognormal(np.log(407.0), 0.66)), 200, 4000))
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        if i % 3 == 0:
            w = rng.choice(22, size=int(rng.integers(60, 81)), p=prd).astype(np.uint8)
            a, b = np.sort(rng.choice(n - len(w), size=2, replace=False))
            s[a:a + len(w)] = w
            s[b:b + len(w)] = w
        elif i % 3 == 1:
            w = rng.choice(22, size=60, p=prd).astype(np.uint8)
            a, b = np.sort(rng.choice(n - 60, size=2, replace=False))
            s[a:a + 60] = w
            s[b:b + 60] = rng.permutation(w)
        else:
            m = rng.choice(22, size=int(rng.integers(4, 12)), p=prd).astype(np.uint8)
            a = int(rng.integers(0, n - 80))
            s[a:a + 80] = np.resize(m, 80)
        seqs.append(s)
    lens = np.array([len(x) for x in seqs], dtype=np.int64)
    offsets = np.zeros(nprot + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return np.concatenate(seqs), offsets


def edge_cases(seed=7):
    """Ragged / degenerate inputs: n = 1..3, around the window (20/21/40/41/42) and core
    (59/60/61) and MW (79/80/81) sizes, all-X, poly-Q, poly-P (PAPA proline rule), stop codons inside."""
    rng = np.random.default_rng(seed)
    seqs = []
    for n in [1, 2, 3, 4, 5, 6, 9, 10, 19, 20, 21, 22, 39, 40, 41, 42, 43, 59, 60, 61, 62, 79, 80, 81, 82, 83, 84,
              100, 101, 120, 121, 122, 123, 127, 128, 129, 255, 256, 257]:
        seqs.append(rng.integers(1, 21, size=n).astype(np.uint8))
        seqs.append(rng.choice(22, size=n, p=PRD_28 / PRD_28.sum()).astype(np.uint8))
    seqs.append(np.zeros(150, np.uint8))                     # all X
    seqs.append(np.full(200, 14, np.uint8))                  # poly-Q (exact plateaus / ties)
    seqs.append(np.full(130, 13, np.uint8))                  # poly-P
    seqs.append(np.tile(np.array([13, 1, 13, 13, 12], np.uint8), 40))  # P.P / PP patterns
    seqs.append(np.tile(np.array([14, 12], np.uint8), 120))  # (QN)n periodic ties
    s = rng.integers(1, 21, size=300).astype(np.uint8)
    s[[0, 5, 150, 299]] = 21                                 # '*' inside and at position 0 / last-but-stripped
    seqs.append(s)
    s = rng.choice(22, size=700, p=BG_SCER / BG_SCER.sum()).astype(np.uint8)
    s[300:420] = rng.choice(22, size=120, p=PRD_28 / PRD_28.sum())
    seqs.append(s)                                           # a clear PrD in the middle
    s = rng.choice(22, size=400, p=PRD_28 / PRD_28.sum()).astype(np.uint8)
    seqs.append(s)                                           # PrD end to end
    lens = np.array([len(x) for x in seqs], dtype=np.int64)
    offsets = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return np.concatenate(seqs).astype(np.uint8), offsets

# web/bg_freqs/bg_freqs_HUMAN.txt of the reference (UniProt human proteome residue counts; data, X..*)
BG_HUMAN_COUNTS = np.array([6721, 2428201, 765477, 1681675, 2518353, 1243278, 2277183, 901810, 1518152, 2016587,
                            3445627, 764646, 1257376, 2211452, 1685966, 1984919, 2928531, 1884442, 2097434, 430493,
                            910830, 0], dtype=np.float64)


def long_proteins(seed=1005, lengths=(35000, 100000)):
    """Config 5: titin-length and 100k-aa proteins, background composition with 150-aa PrD-like
    segments at 10 %, 50 % and 86 % of the length (the late one exercises the -1e6 mask pollution)."""
    rng = np.random.default_rng(seed)
    seqs = []
    for n in lengths:
        s = rng.choice(22, size=n, p=BG_SCER / BG_SCER.sum()).astype(np.uint8)
        for frac in (0.10, 0.50, 0.86):
            st = int(n * frac)
            s[st:st + 150] = rng.choice(22, size=150, p=PRD_28 / PRD_28.sum())
        seqs.append(s)
    lens = np.array([len(x) for x in seqs], dtype=np.int64)
    offsets = np.zeros(len(seqs) + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    return np.concatenate(seqs), offsets
