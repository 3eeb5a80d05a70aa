"""Shuffle nulls (plaac_score_shuffles) against scoring the same replicates device-resident and from pinned host buffers.

Workloads (references from variants_bench.workloads()):
  (a) the yeast-sized reference (5 880 proteins) x K = 1 000, about 3e9 replicate residues;
  (b) 1 000 proteins of bench.py's length distribution x K = 1 000;
  (c) one 34 000-residue protein x K = 10 000 (latency-bound, as the variant scan of that protein).
For each: the wall time of the null call (3 default columns, counts only) from pinned host buffers (host clock around
the blocking call, median of 3), and, on a materialised sample of the first replicates (about 4e8 residues, built with
plaac_shuffle_host), plaac_score_device (codes already resident) and plaac_score from pinned host buffers, the three
alternating so that drift in the machine affects them alike.  The rate of each is in replicate residues/s.  A separate
torch.profiler run gives the device time of the expansion and tally kernels next to the summary kernel.  The sample's
records are checked against the call's values.

Usage: python scripts/gpu/shuffle_null_bench.py [--out profiles/shuffle_null_bench.json] [--sample-res 4e8]
"""
import argparse
import json
import os
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import plaac_b200  # noqa: E402
from variants_bench import card, pinned, workloads  # noqa: E402

REPS = 3
SEED = 11
COLS = ("llr", "core_score", "hmm_all")


def materialise(codes, offsets, K, nrep):
    """Replicates q = 0 .. nrep-1 (q = i*K + r) as an ordinary batch, built on all host threads."""
    q = np.arange(nrep, dtype=np.int64)
    prot = q // K
    lens = offsets[prot + 1] - offsets[prot]
    off = np.zeros(nrep + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    mc = np.empty(int(off[-1]), dtype=np.uint8)
    L = plaac_b200.lib()

    def part(lo, hi):
        for t in range(lo, hi):
            i = int(prot[t])
            src = codes[offsets[i]:offsets[i + 1]]
            rc = L.plaac_shuffle_host(src.ctypes.data, len(src), SEED, i, int(q[t] - i * K), mc[off[t]:].ctypes.data)
            assert rc == 0

    nt = max(1, min(64, os.cpu_count() or 1))
    step = (nrep + nt - 1) // nt
    with ThreadPoolExecutor(nt) as ex:
        list(ex.map(lambda a: part(a, min(nrep, a + step)), range(0, nrep, step)))
    return mc, off


def profile_kernels(sc, codes, offsets, K):
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sc.shuffle_null(codes, offsets, K, seed=SEED, columns=COLS)
            torch.cuda.synchronize()
        out, total = {}, 0.0
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = getattr(e, "self_cuda_time_total", 0.0)
            t = float(t) / 1e3  # us -> ms
            if e.key.startswith("k_") or "plaac" in e.key or "void" in e.key:
                total += t
            for k in ("k_shuffle_prep", "k_shuffle_expand", "k_shuffle_tally", "k_score_summary", "k_long", "k_pack"):
                if k in e.key:
                    out[k] = out.get(k, 0.0) + t
        return {"ms": out, "all_kernels_ms": total}
    except Exception as e:  # noqa: BLE001
        return {"error": f"not measured: {e}"}


def run_workload(name, codes, offsets, K, sample_res):
    import torch

    keep = []
    nprot = len(offsets) - 1
    lens = np.diff(offsets)
    nres = int(lens.sum()) * K
    pc, po = pinned(codes, keep), pinned(offsets, keep)
    sc = plaac_b200.Scorer()
    # (a pinned counts array, so the call's own output needs no staging)
    counts = plaac_b200.PinnedBuffer(nprot, dtype=[(n, "<i8") for n in COLS])
    keep.append(counts)
    mask = sum(1 << plaac_b200.NULL_COLUMNS.index(c) for c in COLS)

    def call():
        import ctypes as C

        nl = plaac_b200.Null(replicates=K, seed=SEED, columns=mask, reserved=0, nsel=-1, proteins=None,
                             counts=counts.array.ctypes.data, values=None)
        rc = plaac_b200.lib().plaac_score_shuffles(sc._h, pc.ctypes.data, po.ctypes.data, nprot, C.byref(nl), None)
        assert rc == 0, plaac_b200.lib().plaac_last_error(sc._h).decode()

    # the materialised sample: the first replicates up to sample_res residues
    cum = np.cumsum(np.repeat(lens, K)) if nprot * K <= 50_000_000 else None
    if cum is not None:
        nrep = int(np.searchsorted(cum, sample_res, side="right"))
    else:
        nrep = int(sample_res // max(1, lens.mean()))
    nrep = max(1, min(nprot * K, nrep))
    t0 = time.perf_counter()
    mc, mo = materialise(codes, offsets, K, nrep)
    t_mat = time.perf_counter() - t0
    sres = int(mo[-1])
    base = plaac_b200.Scorer()
    base.set_long_path(-1)
    dc = torch.from_numpy(mc).cuda()
    do = torch.from_numpy(mo).cuda()
    dsum = torch.zeros(nrep * 160, dtype=torch.uint8, device="cuda")
    mpc, mpo = pinned(mc, keep), pinned(mo, keep)
    hout = plaac_b200.PinnedBuffer(nrep, dtype=plaac_b200.SUMMARY_DTYPE)
    keep.append(hout)

    ways = {
        "null_call": call,
        "device_resident": lambda: base.score_device(dc.data_ptr(), do.data_ptr(), nrep, sres, dsum.data_ptr()),
        "host_pinned_plaac_score": lambda: base.score_ptr(mpc.ctypes.data, mpo.ctypes.data, nrep, hout.array.ctypes.data),
    }
    for f in ways.values():
        f()  # warm-up: every buffer allocated
    times = {w: [] for w in ways}
    for _ in range(REPS):
        for w, f in ways.items():
            t0 = time.perf_counter()
            f()  # (each ends in a synchronise)
            times[w].append(time.perf_counter() - t0)
    # the sample's records against the call's values
    _, vals = sc.shuffle_null(codes, offsets, K, seed=SEED, columns=COLS, values=True)
    v = vals.reshape(-1)[:nrep]
    rec = hout.array
    same = all(np.array_equal(np.ascontiguousarray(v[c]).view(np.uint64), np.ascontiguousarray(rec[c]).view(np.uint64))
               for c in COLS)
    same &= bool((dsum.cpu().numpy().view(np.uint8) == rec.view(np.uint8)).all())
    del vals, v
    kern = profile_kernels(sc, pc, po, K)
    sc.close()
    base.close()
    r = {"workload": name, "proteins": nprot, "replicates": K, "replicate_residues": nres, "total_replicates": nprot * K}
    med = {w: float(np.median(t)) for w, t in times.items()}
    r["null_call"] = {"wall_s": times["null_call"], "wall_s_median": med["null_call"],
                      "residues_per_s": nres / med["null_call"], "h2d_bytes": codes.nbytes + offsets.nbytes + 160 * nprot,
                      "d2h_bytes": 8 * len(COLS) * nprot + 160 * nprot}
    r["sample"] = {"replicates": nrep, "residues": sres, "host_build_s": t_mat, "records_equal_to_call_values": bool(same)}
    for w in ("device_resident", "host_pinned_plaac_score"):
        r["sample"][w] = {"wall_s": times[w], "residues_per_s": sres / med[w]}
    r["call_rate_over_device_resident"] = r["null_call"]["residues_per_s"] / r["sample"]["device_resident"]["residues_per_s"]
    r["kernels"] = kern
    del dc, do, dsum
    for b in keep:
        b.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "shuffle_null_bench.json"))
    ap.add_argument("--sample-res", type=float, default=4e8)
    a = ap.parse_args()
    if plaac_b200.lib().plaac_device_count() <= 0:
        sys.exit("shuffle_null_bench: no CUDA device")
    info = {"card": card(), "timing": "host clock around the blocking call, median of 3, alternating with the baselines",
            "columns": list(COLS), "seed": SEED, "results": []}
    print("card:", info["card"], flush=True)
    wl = {n[0]: (c, o) for n, c, o, _ in workloads()}
    plan = [("a: yeast-sized reference (5 880 proteins) x K = 1 000", wl["c"], 1000),
            ("b: 1 000 bench-distribution proteins x K = 1 000", wl["b"], 1000),
            ("c: one 34 000-residue protein x K = 10 000", wl["a"], 10000)]
    for name, (c, o), K in plan:
        r = run_workload(name, c, o, K, a.sample_res)
        info["results"].append(r)
        s = r["sample"]
        print(f"{name}: call {r['null_call']['wall_s_median'] * 1e3:.1f} ms = {r['null_call']['residues_per_s']:.3g} res/s; "
              f"device-resident {s['device_resident']['residues_per_s']:.3g}; pinned plaac_score "
              f"{s['host_pinned_plaac_score']['residues_per_s']:.3g}; ratio {r['call_rate_over_device_resident']:.2f}; "
              f"kernels {r['kernels']}; equal {s['records_equal_to_call_values']}", flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
