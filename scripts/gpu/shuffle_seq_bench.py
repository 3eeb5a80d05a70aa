"""Sequential shuffle nulls (plaac_score_shuffles_seq) against the fixed call (plaac_score_shuffles) at the same K_max.

Workloads (references from variants_bench.workloads()), h = 10, the three default columns, pinned host buffers:
  (a)  the yeast-sized reference (5 880 proteins) x K_max = 1e5; the fixed call at K = 1e5 is measured once (about 7 s);
  (a') the same x K_max = 1e6; the fixed call's time is extrapolated from (a) (x 10), not measured;
  (b)  1 000 proteins of bench.py's length distribution x K_max = 1e5, against the fixed call at K = 1e5;
  (c)  one 34 000-residue protein x K_max = 1e4, against the fixed call at K = 1e4.
Times are a host clock around the blocking call, median of 3, the sequential call alternating with the fixed one.  For
the sequential call: its rounds, the sum of L over proteins and columns, and the replicate residues the GPU scored,
worked out from the documented schedule (DESIGN.md section 14): protein j is scored up to the first round bound R_g at or
above its largest L ("rounds" counts the bounds the schedule reaches).  The rate of either call is replicate residues
scored per second.  A separate torch.profiler run of (a) gives the device time of the round kernels next to the
expansion and summary kernels.

Usage: python scripts/gpu/shuffle_seq_bench.py [--out profiles/shuffle_seq_bench.json]
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
CHUNK_RES = 256 << 20  # the library's default chunk bound, from which the flag budget derives


def bounds(lens, last, h, K, k):
    """R_1, R_2, ... of DESIGN.md section 14 at the default chunk bound; last[j] = the largest L of protein j (it stays
    active after R_g while last[j] > R_g)."""
    wcap = max(CHUNK_RES // 32, k) // k * 32
    out, r, active = [], 0, np.ones(len(lens), dtype=bool)
    while active.any() and r < K:
        res = max(int(lens[active].sum()), 1)
        wmin = -(-CHUNK_RES // res)
        w = min(K - r, max(r if r else (K if h > K // 4 else max(64, 4 * h)), wmin))
        if K - r - w < wmin:
            w = K - r
        r += min(w, wcap)
        out.append(r)
        active &= last > r
    return np.array(out, dtype=np.int64)


class Calls:
    def __init__(self, codes, offsets):
        self.keep = []
        self.nprot = len(offsets) - 1
        self.pc, self.po = pinned(codes, self.keep), pinned(offsets, self.keep)
        dt = [(n, "<i8") for n in COLS]
        self.counts = plaac_b200.PinnedBuffer(self.nprot, dtype=dt)
        self.scored = plaac_b200.PinnedBuffer(self.nprot, dtype=dt)
        self.fixed_counts = plaac_b200.PinnedBuffer(self.nprot, dtype=dt)  # (the alternating calls keep their own)
        self.keep += [self.counts, self.scored, self.fixed_counts]
        self.sc = plaac_b200.Scorer()

    def _null(self, K, counts):
        return plaac_b200.Null(replicates=K, seed=SEED, columns=MASK, reserved=0, nsel=-1, proteins=None,
                               counts=counts.array.ctypes.data, values=None)

    def fixed(self, K):
        nl = self._null(K, self.fixed_counts)
        rc = plaac_b200.lib().plaac_score_shuffles(self.sc._h, self.pc.ctypes.data, self.po.ctypes.data, self.nprot,
                                                   C.byref(nl), None)
        assert rc == 0, plaac_b200.lib().plaac_last_error(self.sc._h).decode()

    def seq(self, K):
        nl = self._null(K, self.counts)
        rc = plaac_b200.lib().plaac_score_shuffles_seq(self.sc._h, self.pc.ctypes.data, self.po.ctypes.data, self.nprot,
                                                       C.byref(nl), H, self.scored.array.ctypes.data, None)
        assert rc == 0, plaac_b200.lib().plaac_last_error(self.sc._h).decode()

    def close(self):
        self.sc.close()
        for b in self.keep:
            b.close()


def timed(f, *a):
    t0 = time.perf_counter()
    f(*a)  # (blocks until done)
    return time.perf_counter() - t0


def profile_kernels(calls, K):
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            calls.seq(K)
            torch.cuda.synchronize()
        out, total = {}, 0.0
        names = ("k_shuffle_flags", "k_shuffle_stop", "k_shuffle_compact", "k_scan", "k_shuffle_prep", "k_shuffle_expand",
                 "k_score_summary", "k_long", "k_pack")
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = getattr(e, "self_cuda_time_total", 0.0)
            t = float(t) / 1e3  # us -> ms
            if e.key.startswith("k_") or "plaac" in e.key or "void" in e.key:
                total += t
            for k in names:
                if k in e.key:
                    out[k] = out.get(k, 0.0) + t
        return {"ms": out, "all_kernels_ms": total}
    except Exception as e:  # noqa: BLE001
        return {"error": f"not measured: {e}"}


def run_workload(name, codes, offsets, K, fixed_reps, fixed_from=None, profile=False):
    calls = Calls(codes, offsets)
    lens = np.diff(offsets).astype(np.int64)
    calls.seq(min(K, 1000))  # warm-up: every buffer allocated
    calls.fixed(1000)
    t_seq, t_fix = [], []
    for rep in range(REPS):
        t_seq.append(timed(calls.seq, K))
        if rep < fixed_reps:
            t_fix.append(timed(calls.fixed, K))
    L = np.stack([calls.scored.array[c] for c in COLS], axis=1)
    n = np.stack([calls.counts.array[c] for c in COLS], axis=1)
    R = bounds(lens, L.max(axis=1), H, K, len(COLS))
    g = np.searchsorted(R, L.max(axis=1), side="left")  # the round in which the protein's last column stopped
    reps = R[g]
    r = {"workload": name, "proteins": int(len(lens)), "K_max": K, "stop_hits": H}
    med = float(np.median(t_seq))
    scored_res = int((lens * reps).sum())
    r["seq"] = {"wall_s": t_seq, "wall_s_median": med, "rounds": len(R), "round_bounds": R.tolist(),
                "sum_L": int(L.sum()), "columns_stopped": int((n == H).sum()), "columns": int(n.size),
                "replicates_scored": int(reps.sum()), "replicate_residues_scored": scored_res,
                "residues_per_s": scored_res / med}
    full = int(lens.sum()) * K
    if t_fix:
        fm = float(np.median(t_fix))
        r["fixed"] = {"wall_s": t_fix, "wall_s_median": fm, "measured": True, "replicate_residues": full,
                      "residues_per_s": full / fm}
    else:
        base = fixed_from["fixed"]
        fm = base["wall_s_median"] * K / fixed_from["K_max"]
        r["fixed"] = {"wall_s_median": fm, "measured": False,
                      "extrapolated_from": f"{fixed_from['workload']} x {K // fixed_from['K_max']}",
                      "replicate_residues": full, "residues_per_s": base["residues_per_s"]}
    r["speedup_over_fixed"] = fm / med
    r["rate_seq_over_fixed"] = r["seq"]["residues_per_s"] / r["fixed"]["residues_per_s"]
    if profile:
        r["kernels"] = profile_kernels(calls, K)
    calls.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shuffle_seq_bench.json"))
    a = ap.parse_args()
    if plaac_b200.lib().plaac_device_count() <= 0:
        sys.exit("shuffle_seq_bench: no CUDA device")
    info = {"card": card(), "timing": "host clock around the blocking call, median of 3, alternating with the fixed call",
            "columns": list(COLS), "seed": SEED, "stop_hits": H, "results": []}
    print("card:", info["card"], flush=True)
    wl = {n[0]: (c, o) for n, c, o, _ in workloads()}
    ra = run_workload("a: yeast-sized reference (5 880 proteins) x K_max = 1e5", *wl["c"], 100_000, 1, profile=True)
    rows = [ra,
            run_workload("a': yeast-sized reference x K_max = 1e6", *wl["c"], 1_000_000, 0, fixed_from=ra),
            run_workload("b: 1 000 bench-distribution proteins x K_max = 1e5", *wl["b"], 100_000, REPS),
            run_workload("c: one 34 000-residue protein x K_max = 1e4", *wl["a"], 10_000, REPS)]
    for r in rows:
        info["results"].append(r)
        s, f = r["seq"], r["fixed"]
        print(f"{r['workload']}: seq {s['wall_s_median'] * 1e3:.1f} ms ({s['rounds']} rounds, {s['replicates_scored']} "
              f"replicates, {s['residues_per_s']:.3g} res/s); fixed {f['wall_s_median'] * 1e3:.1f} ms "
              f"({'measured' if f['measured'] else 'extrapolated'}, {f['residues_per_s']:.3g} res/s); speedup "
              f"{r['speedup_over_fixed']:.1f}; rate ratio {r['rate_seq_over_fixed']:.2f}", flush=True)
    print("kernels (a):", ra.get("kernels"), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
