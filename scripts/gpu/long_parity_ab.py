"""Byte-for-byte comparison of the long-sequence path between two source trees (a refactor must not change one byte).

    cd TREE_A && python /path/to/long_parity_ab.py dump /tmp/a.npz     # run inside each tree: its plaac_b200 is used
    cd TREE_B && python /path/to/long_parity_ab.py dump /tmp/b.npz
    python long_parity_ab.py compare /tmp/a.npz /tmp/b.npz
    python long_parity_ab.py compare-dirs DIR_A DIR_B                  # two bench.py --dump-outputs directories

`dump` scores, with records only, with records and per-residue arrays, and with per-residue arrays only:
  * synth.long_proteins() (35 k and 100 k residues), fixed threshold 8192;
  * the mixed batch of test_long_path_mixed_batch_thresholds_and_fallback (lengths around the chunk geometry, 800 short
    proteins) with set_long_path at 1024, 4096, -1 (automatic) and 0 (off), and at 1024 with warm-ups -1 and 3;
  * a yeast-sized set of 6 000 proteins with the automatic threshold.
It keeps every record byte, a SHA-256 of every per-residue array and the long-path counters of each run.
"""
import hashlib
import os
import sys

import numpy as np

sys.path.insert(0, os.getcwd())  # the tree being measured, not the one this file lives in


def mixed_batch():
    from tests import synth
    import plaac_b200

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
            s[-200:] = rng.choice(22, size=200, p=prd)
        seqs.append(s)
    seqs.append(np.full(5000, 14, np.uint8))
    seqs.append(np.tile(np.array([13, 1, 13, 13, 12], np.uint8), 1200))
    seqs.append(rng.integers(1, 21, size=6000).astype(np.uint8))
    c2, o2 = synth.proteome(800, seed=5)
    seqs += [c2[o2[i]:o2[i + 1]] for i in range(800)]
    order = rng.permutation(len(seqs))
    return plaac_b200.pack([seqs[i] for i in order])


def dump(path):
    import plaac_b200
    from tests import synth

    runs = [("long", synth.long_proteins(), [(8192, 0)]),
            ("mixed", mixed_batch(), [(1024, 0), (4096, 0), (-1, 0), (0, 0), (1024, -1), (1024, 3)]),
            ("yeast6k", synth.proteome(6000, seed=2024), [(-1, 0)])]
    out = {}
    for name, (codes, offs), settings in runs:
        for min_len, warm in settings:
            for mode in ("rec", "rec+res", "res"):
                sc = plaac_b200.Scorer(device=0)
                sc.set_long_path(min_len, warm)
                if mode == "rec":
                    rec, res = sc.score(codes, offs), None
                elif mode == "rec+res":
                    rec, res = sc.score(codes, offs, per_residue=True)
                else:
                    rec, res = sc.score(codes, offs, per_residue=True, summaries=False)
                st = sc.stats()
                sc.close()
                key = f"{name}/{min_len}/{warm}/{mode}"
                if rec is not None:
                    out[key + "/records"] = np.frombuffer(rec.tobytes(), np.uint8)
                for k, a in sorted((res or {}).items()):
                    out[key + "/" + k] = np.frombuffer(hashlib.sha256(a.tobytes()).digest(), np.uint8)
                out[key + "/counters"] = np.array([st.long_proteins, st.long_redone_chunks], np.int64)
                print(key, "long proteins", st.long_proteins, "redone chunks", st.long_redone_chunks, flush=True)
    np.savez(path, **out)


def compare(a_path, b_path):
    a, b = np.load(a_path), np.load(b_path)
    bad = sorted(set(a.files) ^ set(b.files))
    for k in sorted(set(a.files) & set(b.files)):
        if a[k].tobytes() != b[k].tobytes():
            bad.append(k)
    print(f"{len(a.files)} arrays compared, {len(bad)} differ" + "".join("\n  " + k for k in bad))
    return not bad


def compare_dirs(a_dir, b_dir):
    fa, fb = sorted(os.listdir(a_dir)), sorted(os.listdir(b_dir))
    bad = sorted(set(fa) ^ set(fb))
    for f in sorted(set(fa) & set(fb)):
        if np.load(os.path.join(a_dir, f)).tobytes() != np.load(os.path.join(b_dir, f)).tobytes():
            bad.append(f)
    print(f"{len(fa)} arrays compared, {len(bad)} differ" + "".join("\n  " + f for f in bad))
    return not bad


if __name__ == "__main__":
    cmd = sys.argv[1]
    if cmd == "dump":
        dump(sys.argv[2])
    else:
        ok = (compare if cmd == "compare" else compare_dirs)(sys.argv[2], sys.argv[3])
        sys.exit(0 if ok else 1)
