"""Variant effects (plaac_score_variant_effects) against whole records (plaac_score_variants).

The three workloads of variants_bench.py, each scored three ways from pinned host buffers into a pinned output:
effects with 1 column (core_score), effects with 3 columns (core_score, llr, core_change), and the full records.  Each
is timed with the host clock around the blocking call, median of 3, the three ways alternating so that drift in the
machine affects them alike.  The bytes each way moves over the host link are counted from the array sizes.  The
effect call also scores the reference once (its records go to the host and back up into the device table), so that
traffic is counted too.  The effects are checked against the records minus plaac_score's wild-type records.

Usage: python scripts/gpu/variant_effects_bench.py [--out profiles/variant_effects_bench.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import plaac_b200  # noqa: E402
from variants_bench import card, pinned, workloads  # noqa: E402

REPS = 3
WAYS = {"effects_1": ("core_score",), "effects_3": ("core_score", "llr", "core_change"), "records": None}


def run_workload(name, codes, offsets, var):
    keep = []
    nvar = len(var[0])
    nref = len(offsets) - 1
    nsub = int(var[1][-1])
    lens = offsets[var[0].astype(np.int64) + 1] - offsets[var[0].astype(np.int64)]
    nres = int(lens.sum())
    args = [pinned(codes, keep), pinned(offsets, keep)] + [pinned(x, keep) for x in var]
    outs = {}
    for way, cols in WAYS.items():
        dt = plaac_b200.SUMMARY_DTYPE if cols is None else plaac_b200.effects_dtype(
            sum(1 << plaac_b200.EFFECT_COLUMNS.index(c) for c in cols))
        outs[way] = plaac_b200.PinnedBuffer(nvar, dtype=dt)
        keep.append(outs[way])
    sc = plaac_b200.Scorer()

    def call(way):
        if WAYS[way] is None:
            sc.score_variants(*args, out=outs[way].array)
        else:
            sc.variant_effects(*args, columns=WAYS[way], out=outs[way].array)

    for way in WAYS:
        call(way)  # warm-up: every buffer allocated
    times = {w: [] for w in WAYS}
    for _ in range(REPS):
        for way in WAYS:
            t0 = time.perf_counter()
            call(way)
            times[way].append(time.perf_counter() - t0)
    # the part of the effect call that does not grow with the variants: one plain scoring of the reference
    t_ref = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        wt = sc.score(args[0], args[1])
        t_ref.append(time.perf_counter() - t0)
    sc.close()
    rec = outs["records"].array
    w = wt[var[0].astype(np.int64)]
    with np.errstate(invalid="ignore"):
        want = {"core_score": rec["core_score"] - w["core_score"], "llr": rec["llr"] - w["llr"],
                "core_change": (~np.isnan(rec["core_score"])).astype(float) - (~np.isnan(w["core_score"])).astype(float)}
    equal = True
    for way in ("effects_1", "effects_3"):
        e = outs[way].array
        for c in e.dtype.names:
            g, x = np.ascontiguousarray(e[c]), want[c]
            equal &= bool(np.array_equal(np.isnan(g), np.isnan(x)) and
                          (g.view(np.uint64) == x.view(np.uint64))[~np.isnan(x)].all())
    # host link traffic: the variant list and the reference as plaac_score_variants moves them; the effect call adds one
    # plain scoring of the reference (codes and offsets up, records down) and the upload of those records
    h2d = codes.nbytes + offsets.nbytes + 4 * nvar + 8 * (nvar + 1) + 5 * nsub
    r = {"workload": name, "variants": nvar, "reference_proteins": nref, "variant_residues": nres}
    for way, cols in WAYS.items():
        med = float(np.median(times[way]))
        if cols is None:
            link = {"h2d_bytes": h2d, "d2h_bytes": 160 * nvar}
        else:
            link = {"h2d_bytes": h2d + codes.nbytes + offsets.nbytes + 160 * nref,
                    "d2h_bytes": 8 * len(cols) * nvar + 160 * nref}
        r[way] = {"columns": list(cols) if cols else None, "wall_s": times[way], "wall_s_median": med,
                  "residues_per_s": nres / med, **link}
    r["reference_plaac_score_s"] = t_ref
    r["effects_equal_records_minus_wild"] = equal
    for b in keep:
        b.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "variant_effects_bench.json"))
    a = ap.parse_args()
    if plaac_b200.lib().plaac_device_count() <= 0:
        sys.exit("variant_effects_bench: no CUDA device")
    info = {"card": card(), "timing": "host clock around the blocking call from pinned host buffers, median of 3",
            "results": []}
    print("card:", info["card"], flush=True)
    for name, c, o, var in workloads():
        r = run_workload(name, c, o, var)
        info["results"].append(r)
        print(name + ": " + "; ".join(f"{w} {r[w]['wall_s_median'] * 1e3:.1f} ms (D2H {r[w]['d2h_bytes'] / 1e6:.1f} MB)"
                                      for w in WAYS) + f"; reference alone {np.median(r['reference_plaac_score_s']) * 1e3:.1f} ms"
              + f"; effects equal: {r['effects_equal_records_minus_wild']}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
