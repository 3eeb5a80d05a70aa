"""Prion-like segments (plaac_score_segments) against what they add to, and against the route they replace.

  (a) plaac_score against plaac_score_segments (records and segments) on a bench-distribution batch of at least 2e9
      residues (bench.synth_shard) and on a yeast-sized set;
  (b) the same two calls on one 100 000-residue protein, which takes the long path;
  (c) on 200 000 bench-distribution proteins, plaac_score_segments against the per-residue route: plaac_score with only
      the VIT column requested, then the runs and their scores found on the host (vectorised numpy).

Every call reads and writes pinned host buffers and is timed with the host clock around the blocking call, median of 3,
the ways alternating so that drift in the machine affects them alike.  The segments of each way are checked against
each other.  A separate torch.profiler run records the kernel durations of one plaac_score_segments call per workload.

Usage: python scripts/gpu/segments_bench.py [--out profiles/segments_bench.json]
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

import bench  # noqa: E402
import plaac_b200  # noqa: E402
from tests import synth  # noqa: E402
from variants_bench import card, pinned  # noqa: E402

REPS = 3


def bench_batch(nprot):
    import torch

    codes, offsets, ntotal = bench.synth_shard(plaac_b200.lib(), torch.device("cuda", 0), 0, nprot)
    torch.cuda.synchronize()
    h_codes, h_offs = codes[:ntotal].cpu().numpy(), offsets.cpu().numpy()
    del codes, offsets
    torch.cuda.empty_cache()
    return h_codes, h_offs


class Ways:
    """Pinned inputs and outputs of one workload, and the calls."""

    def __init__(self, codes, offsets, cap):
        self.keep = []
        self.nprot = len(offsets) - 1
        self.nres = int(offsets[-1] - offsets[0])
        self.codes = pinned(codes, self.keep)
        self.offs = pinned(offsets, self.keep)
        self.rec = self.buf(self.nprot, plaac_b200.SUMMARY_DTYPE)
        self.first = self.buf(self.nprot + 1, np.int64)
        self.cap = cap
        self.start, self.end = self.buf(cap, np.int32), self.buf(cap, np.int32)
        self.score = self.buf(cap, np.float64)
        self.sc = plaac_b200.Scorer()
        self.count = 0

    def buf(self, n, dt):
        b = plaac_b200.PinnedBuffer(max(int(n), 1), dtype=dt)
        self.keep.append(b)
        return b

    def call_score(self):
        self.sc._check(plaac_b200.lib().plaac_score(self.sc._h, self.codes.ctypes.data, self.offs.ctypes.data, self.nprot,
                                                    self.rec.ptr, None))

    def call_segments(self):
        g = plaac_b200.Segments(capacity=self.cap, first=self.first.ptr, start=self.start.ptr, end=self.end.ptr,
                                score=self.score.ptr, count=0)
        self.sc._check(plaac_b200.lib().plaac_score_segments(self.sc._h, self.codes.ctypes.data, self.offs.ctypes.data,
                                                             self.nprot, self.rec.ptr, C.byref(g)))
        assert g.count <= self.cap, (g.count, self.cap)
        self.count = int(g.count)

    def result(self):
        n = self.count
        return {"first": self.first.array.copy(), "start": self.start.array[:n].copy(), "end": self.end.array[:n].copy(),
                "score": self.score.array[:n].copy()}

    def close(self):
        self.sc.close()
        for b in self.keep:
            b.close()


def timed(fns):
    for f in fns.values():
        f()  # warm-up: every buffer allocated
    t = {k: [] for k in fns}
    for _ in range(REPS):
        for k, f in fns.items():
            t0 = time.perf_counter()
            f()
            t[k].append(time.perf_counter() - t0)
    return t


def summary_vs_segments(name, codes, offsets, cap):
    w = Ways(codes, offsets, cap)
    t = timed({"plaac_score": w.call_score, "plaac_score_segments": w.call_segments})
    r = {"workload": name, "proteins": w.nprot, "residues": w.nres, "segments": w.count}
    for k, v in t.items():
        r[k] = {"wall_s": v, "wall_s_median": float(np.median(v)), "residues_per_s": w.nres / float(np.median(v))}
    r["segments_over_score"] = r["plaac_score_segments"]["wall_s_median"] / r["plaac_score"]["wall_s_median"]
    r["kernels_us"] = kernel_times(w.call_segments)
    w.close()
    return r


def host_runs(codes, offsets, vit, llr):
    """The per-residue route's host side: runs of 1s of the VIT column that stay inside a protein, and their llr sums."""
    v = vit.astype(np.int8)
    nres = len(v)
    brk = np.zeros(nres + 1, dtype=bool)
    brk[(offsets[1:-1] - offsets[0]).astype(np.int64)] = True
    prev = np.r_[np.int8(0), v[:-1]]
    prev[brk[:-1]] = 0
    starts = np.nonzero((v == 1) & (prev == 0))[0]
    nxt = np.r_[v[1:], np.int8(0)]
    nxt[brk[1:]] = 0
    ends = np.nonzero((v == 1) & (nxt == 0))[0]
    vals = np.r_[llr[np.where(codes > 21, 0, codes)], 0.0]
    # sums over [start, end]: reduceat over start, end + 1 pairs, every other result (numpy sums a block pairwise, so
    # these are not PRDscore's bits; the route is timed, and compared on first / start / end only)
    score = np.add.reduceat(vals, np.ravel(np.c_[starts, ends + 1]))[::2] if len(starts) else np.zeros(0)
    prot = np.searchsorted(offsets - offsets[0], starts, side="right") - 1
    first = np.searchsorted(prot, np.arange(len(offsets)), side="left")
    return {"first": first, "start": starts - (offsets[prot] - offsets[0]), "end": ends - (offsets[prot] - offsets[0]),
            "score": score}


def per_residue_route(codes, offsets):
    """(c): plaac_score_segments against plaac_score with only VIT plus the runs found on the host."""
    w = Ways(codes, offsets, len(offsets) - 1)
    vit = w.buf(w.nres, np.uint8)
    ro = plaac_b200.capi.ResidueOut(vit=vit.ptr)
    llr = np.array(w.sc.params.llr[:22], dtype=np.float64)
    out = {}

    def route():
        w.sc._check(plaac_b200.lib().plaac_score(w.sc._h, w.codes.ctypes.data, w.offs.ctypes.data, w.nprot, None, C.byref(ro)))
        out["runs"] = host_runs(w.codes, w.offs, vit.array, llr)

    def route_gpu_only():
        w.sc._check(plaac_b200.lib().plaac_score(w.sc._h, w.codes.ctypes.data, w.offs.ctypes.data, w.nprot, None, C.byref(ro)))

    t = timed({"plaac_score_segments": w.call_segments, "per_residue_vit_plus_host_runs": route,
               "per_residue_vit_call_only": route_gpu_only})
    seg = w.result()
    runs = out["runs"]
    same = (np.array_equal(runs["first"], seg["first"]) and np.array_equal(runs["start"], seg["start"])
            and np.array_equal(runs["end"], seg["end"]))
    r = {"workload": "c: 200 000 bench-distribution proteins", "proteins": w.nprot, "residues": w.nres, "segments": w.count,
         "same_runs": bool(same)}
    for k, v in t.items():
        r[k] = {"wall_s": v, "wall_s_median": float(np.median(v))}
    r["per_residue_over_segments"] = r["per_residue_vit_plus_host_runs"]["wall_s_median"] / r["plaac_score_segments"]["wall_s_median"]
    w.close()
    return r


def kernel_times(fn):
    """Device time per kernel name (microseconds, summed over launches) of one call, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    tot = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            key = e.name.split("(")[0].replace("void ", "").replace("plaac::", "")
            if "k_seg" in key or "k_score_summary" in key or "k_core_search" in key or "k_long" in key or "k_pack" in key:
                tot[key] = tot.get(key, 0.0) + e.device_time
    return {k: round(v, 1) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "segments_bench.json"))
    ap.add_argument("--big-proteins", type=int, default=6_000_000, help="proteins of workload (a)'s large batch")
    a = ap.parse_args()
    if plaac_b200.lib().plaac_device_count() <= 0:
        sys.exit("segments_bench: no CUDA device")
    info = {"card": card(), "timing": "host clock around the blocking call from pinned host buffers, median of 3",
            "results": []}
    print("card:", info["card"], flush=True)

    def report(r):
        info["results"].append(r)
        print(json.dumps({k: (v["wall_s_median"] if isinstance(v, dict) and "wall_s_median" in v else v)
                          for k, v in r.items()}), flush=True)

    codes, offs = bench_batch(a.big_proteins)
    report(summary_vs_segments(f"a: {a.big_proteins} bench-distribution proteins", codes, offs, len(offs) - 1))
    del codes, offs
    codes, offs = synth.proteome(6000, seed=2101)
    report(summary_vs_segments("a: yeast-sized set (6 000 proteins)", codes, offs, len(offs) - 1))
    codes, offs = synth.long_proteins(seed=2102, lengths=(100000,))
    report(summary_vs_segments("b: one 100 000-residue protein (long path)", codes, offs, 1024))
    codes, offs = bench_batch(200_000)
    report(per_residue_route(codes, offs))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
