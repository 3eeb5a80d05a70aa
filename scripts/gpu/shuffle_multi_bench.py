"""Shuffle nulls on several GPUs (plaac_score_shuffles_multi, plaac_score_shuffles_seq_multi) against the single calls.

Workloads (references from variants_bench.workloads()), the three default columns, pinned host buffers:
  (a) the yeast-sized reference (5 880 proteins), fixed call, K = 1e4;
  (b) the same reference, sequential call, K_max = 1e6, h = 10;
  (c) one 34 000-residue protein, sequential call, K_max = 1e5, h = 10 (it never stops: one replicate axis to split).
Each workload runs on N = 1, 2, 4, 8 GPUs (devices 0 .. N-1) as far as the box has them, then with 2 ctxs on device 0,
which gives the cost of the orchestration alone.  Times are a host clock around the blocking call, median of 3, each
multi call alternating with the single call on device 0; the outputs (counts, and L for the sequential call) of every
multi call are checked equal to the single call's, byte for byte.  Parallel efficiency = t_single / (N x t_multi).

Usage: python scripts/gpu/shuffle_multi_bench.py [--out profiles/shuffle_multi_bench.json]
"""
import argparse
import ctypes as C
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
SEED = 11
H = 10
COLS = ("llr", "core_score", "hmm_all")
MASK = sum(1 << plaac_b200.NULL_COLUMNS.index(c) for c in COLS)


class Calls:
    """One workload's pinned inputs and outputs, on a list of ctxs (one ctx: the single call)."""

    def __init__(self, codes, offsets, devices, keep):
        self.nprot = len(offsets) - 1
        self.pc, self.po = pinned(codes, keep), pinned(offsets, keep)
        dt = [(n, "<i8") for n in COLS]
        self.counts = plaac_b200.PinnedBuffer(self.nprot, dtype=dt)
        self.scored = plaac_b200.PinnedBuffer(self.nprot, dtype=dt)
        keep += [self.counts, self.scored]
        self.scorers = [plaac_b200.Scorer(device=d) for d in devices]
        self.hs = (C.c_void_p * len(self.scorers))(*[s._h for s in self.scorers])

    def _null(self, K):
        return plaac_b200.Null(replicates=K, seed=SEED, columns=MASK, reserved=0, nsel=-1, proteins=None,
                               counts=self.counts.array.ctypes.data, values=None)

    def run(self, kind, K):
        nl = self._null(K)
        L = plaac_b200.lib()
        n = len(self.scorers)
        if kind == "fixed":
            rc = L.plaac_score_shuffles_multi(self.hs, n, self.pc.ctypes.data, self.po.ctypes.data, self.nprot, C.byref(nl), None)
        else:
            rc = L.plaac_score_shuffles_seq_multi(self.hs, n, self.pc.ctypes.data, self.po.ctypes.data, self.nprot,
                                                  C.byref(nl), H, self.scored.array.ctypes.data, None)
        assert rc == 0, L.plaac_last_error(self.scorers[0]._h).decode()

    def outputs(self, kind):
        return self.counts.array.tobytes() + (self.scored.array.tobytes() if kind == "seq" else b"")

    def close(self):
        for s in self.scorers:
            s.close()


def timed(calls, kind, K):
    t0 = time.perf_counter()
    calls.run(kind, K)  # (blocks until done)
    return time.perf_counter() - t0


def compare(name, kind, codes, offsets, K, devices, warm):
    """Median of REPS multi calls on `devices`, alternating with the single call on device 0."""
    keep = []
    one = Calls(codes, offsets, [0], keep)
    many = Calls(codes, offsets, devices, keep)
    for c in (one, many):  # warm-up: every buffer allocated, every module loaded
        c.run(kind, warm)
    t1, tn, equal = [], [], True
    for _ in range(REPS):
        t1.append(timed(one, kind, K))
        tn.append(timed(many, kind, K))
        equal &= one.outputs(kind) == many.outputs(kind)
    m1, mn = float(np.median(t1)), float(np.median(tn))
    n = len(devices)
    r = {"workload": name, "call": kind, "K": K, "devices": devices, "single_wall_s": t1, "multi_wall_s": tn,
         "single_wall_s_median": m1, "multi_wall_s_median": mn, "speedup": m1 / mn,
         "parallel_efficiency": m1 / (n * mn) if len(set(devices)) == n else None, "outputs_equal": bool(equal)}
    if kind == "seq":
        r["columns_stopped"] = int(sum((one.counts.array[c] == H).sum() for c in COLS))
        r["sum_L"] = int(sum(one.scored.array[c].sum() for c in COLS))
    one.close()
    many.close()
    for b in keep:
        b.close()
    assert equal, f"{name}, devices {devices}: the multi call's outputs differ from the single call's"
    print(f"{name} on devices {devices}: single {m1 * 1e3:.1f} ms, multi {mn * 1e3:.1f} ms, speedup {m1 / mn:.2f}"
          + (f", efficiency {r['parallel_efficiency']:.2f}" if r["parallel_efficiency"] is not None else ""), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shuffle_multi_bench.json"))
    a = ap.parse_args()
    ndev = plaac_b200.lib().plaac_device_count()
    if ndev <= 0:
        sys.exit("shuffle_multi_bench: no CUDA device")
    ns = [n for n in (1, 2, 4, 8) if n <= ndev]
    info = {"card": card(), "devices_on_box": ndev, "timing": "host clock around the blocking call, median of 3, "
            "alternating with the single call on device 0; outputs checked equal", "columns": list(COLS), "seed": SEED,
            "stop_hits": H, "n_measured": ns, "n_not_measured": [n for n in (1, 2, 4, 8) if n > ndev], "results": []}
    print("card:", info["card"], "devices:", ndev, flush=True)
    wl = {n[0]: (c, o) for n, c, o, _ in workloads()}
    runs = [("a: yeast-sized reference (5 880 proteins), fixed, K = 1e4", "fixed", wl["c"], 10_000, 1000),
            ("b: yeast-sized reference, sequential, K_max = 1e6, h = 10", "seq", wl["c"], 1_000_000, 1000),
            ("c: one 34 000-residue protein, sequential, K_max = 1e5, h = 10", "seq", wl["a"], 100_000, 1000)]
    for name, kind, (codes, offs), K, warm in runs:
        for n in ns:
            info["results"].append(compare(name, kind, codes, offs, K, list(range(n)), warm))
        info["results"].append(compare(name, kind, codes, offs, K, [0, 0], warm))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
