"""Sequence-variant scoring (plaac_score_variants) against the device-resident and the host-buffer path.

Workloads:
  (a) saturation scan of one 34 000-residue synthetic protein (titin-sized; 646 k variants, 2.2e10 residues);
  (b) saturation scan of 1 000 proteins with bench.py's length distribution (lognormal, median 290, sigma 0.62);
  (c) 200 000 random single and double substitutions over a yeast-sized reference (5 880 proteins).
For each: wall time of the variant call from pinned host buffers (host clock around a call that ends in a synchronise)
and its rate in variant residues/s, the bytes it moves over the host link (counted from the array sizes), the kernel
time of the three variant kernels (torch.profiler, a run of its own), and, on a materialised sample of the same variants
that fits in memory, plaac_score_device (codes already resident) and plaac_score from pinned host buffers.  The
baselines use the automatic long-path threshold, as the variant call does.

Usage: python scripts/gpu/variants_bench.py [--out profiles/variants_bench.json] [--sample-res 4e8]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import plaac_b200  # noqa: E402
from tests import synth  # noqa: E402

REPS = 3


def card():
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:  # noqa: BLE001
        return {"name": "unknown", "error": str(e)}


def pinned(a, keep):
    b = plaac_b200.PinnedBuffer(len(a), dtype=a.dtype)
    b.array[:] = a
    keep.append(b)
    return b.array


def materialise(codes, offsets, protein, first_sub, pos, code, lo, hi):
    """Variants [lo, hi) as an ordinary batch."""
    p = protein[lo:hi].astype(np.int64)
    lens = offsets[p + 1] - offsets[p]
    off = np.zeros(len(p) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    idx = np.arange(off[-1], dtype=np.int64) - np.repeat(off[:-1], lens) + np.repeat(offsets[p], lens)
    mc = codes[idx]
    a, b = first_sub[lo], first_sub[hi]
    owner = np.repeat(np.arange(len(p)), np.diff(first_sub[lo:hi + 1]))
    mc[off[owner] + pos[a:b]] = code[a:b]
    return mc, off


def profile_kernels(sc, args):
    try:
        import torch
        from torch.profiler import ProfilerActivity, profile

        torch.cuda.init()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            sc.score_variants(*args)
            torch.cuda.synchronize()
        out, total = {}, 0.0
        for e in prof.key_averages():
            t = getattr(e, "self_device_time_total", None)
            if t is None:
                t = getattr(e, "self_cuda_time_total", 0.0)
            t = float(t) / 1e3  # us -> ms
            if e.key.startswith("k_") or "plaac" in e.key or "void" in e.key:
                total += t
            for k in ("k_variant_lengths", "k_variant_expand", "k_variant_apply"):
                if k in e.key:
                    out[k] = out.get(k, 0.0) + t
        return {"ms": out, "all_kernels_ms": total}
    except Exception as e:  # noqa: BLE001
        return {"error": f"not measured: {e}"}


def run_workload(name, codes, offsets, var, sample_res):
    keep = []
    protein, first_sub, pos, code = var
    nvar = len(protein)
    lens = (offsets[protein.astype(np.int64) + 1] - offsets[protein.astype(np.int64)])
    nres = int(lens.sum())
    args = [pinned(codes, keep), pinned(offsets, keep), pinned(protein, keep), pinned(first_sub, keep), pinned(pos, keep),
            pinned(code, keep)]
    out = plaac_b200.PinnedBuffer(nvar, dtype=plaac_b200.SUMMARY_DTYPE)
    keep.append(out)
    sc = plaac_b200.Scorer()
    sc.score_variants(*args, out=out.array)  # warm-up: every buffer allocated
    times = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        sc.score_variants(*args, out=out.array)
        times.append(time.perf_counter() - t0)
    rec = out.array.copy()
    wall = float(np.median(times))
    nsub = int(first_sub[-1])
    # host -> device: the reference once, then per variant its protein index and first_sub entry, per substitution its
    # position and code (plus one first_sub entry per chunk); device -> host: the records
    h2d = codes.nbytes + offsets.nbytes + 4 * nvar + 8 * (nvar + 1) + 5 * nsub
    d2h = 160 * nvar
    r = {"workload": name, "variants": nvar, "substitutions": nsub, "variant_residues": nres,
         "variant_call": {"wall_s": times, "wall_s_median": wall, "residues_per_s": nres / wall,
                          "h2d_bytes": h2d, "d2h_bytes": d2h, "h2d_bytes_if_materialised": nres + 8 * (nvar + 1)}}
    r["variant_kernels"] = profile_kernels(sc, args + [out.array])
    sc.close()

    # baselines on a materialised sample: the first variants up to sample_res residues
    hi = int(np.searchsorted(np.cumsum(lens), sample_res, side="right"))
    hi = max(1, min(nvar, hi))
    mc, mo = materialise(codes, offsets, protein, first_sub, pos, code, 0, hi)
    sres = int(mo[-1])
    base = plaac_b200.Scorer()
    base.set_long_path(-1)
    import torch

    dc = torch.from_numpy(mc).cuda()
    do = torch.from_numpy(mo).cuda()
    dsum = torch.zeros(hi * 160, dtype=torch.uint8, device="cuda")
    base.score_device(dc.data_ptr(), do.data_ptr(), hi, sres, dsum.data_ptr())
    t_dev = []
    for _ in range(REPS + 2):
        t0 = time.perf_counter()
        base.score_device(dc.data_ptr(), do.data_ptr(), hi, sres, dsum.data_ptr())  # ends in plaac_sync
        t_dev.append(time.perf_counter() - t0)
    dev_rec = dsum.cpu().numpy().view(plaac_b200.SUMMARY_DTYPE)
    pc, po = pinned(mc, keep), pinned(mo, keep)
    hout = plaac_b200.PinnedBuffer(hi, dtype=plaac_b200.SUMMARY_DTYPE)
    keep.append(hout)
    base.score_ptr(pc.ctypes.data, po.ctypes.data, hi, hout.array.ctypes.data)
    t_host = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        base.score_ptr(pc.ctypes.data, po.ctypes.data, hi, hout.array.ctypes.data)
        t_host.append(time.perf_counter() - t0)
    base.close()
    same = bool((rec[:hi].view(np.uint8) == hout.array.view(np.uint8)).all() and
                (dev_rec.view(np.uint8) == hout.array.view(np.uint8)).all())
    r["sample"] = {"variants": hi, "residues": sres, "records_equal_to_variant_call": same,
                   "device_resident": {"wall_s": t_dev, "residues_per_s": sres / float(np.median(t_dev))},
                   "host_pinned_plaac_score": {"wall_s": t_host, "residues_per_s": sres / float(np.median(t_host))}}
    del dc, do, dsum
    for b in keep:
        b.close()
    return r


def workloads():
    """The three workloads of the module docstring: (name, reference codes, reference offsets, variant arrays)."""
    codes, offs = synth.long_proteins(seed=2001, lengths=(34000,))
    wl = [("a: saturation of one 34 000-residue protein", codes, offs, plaac_b200.saturation(codes, offs))]
    codes, offs = synth.proteome(1000, seed=2002, median=290.0, sigma=0.62)
    wl.append(("b: saturation of 1 000 proteins (bench length distribution)", codes, offs, plaac_b200.saturation(codes, offs)))
    codes, offs = synth.proteome(5880, seed=2003)
    rng = np.random.default_rng(2004)
    nvar = 200_000
    protein = rng.integers(0, len(offs) - 1, nvar).astype(np.int32)
    lens = np.diff(offs)[protein]
    nsub = rng.integers(1, 3, nvar)
    nsub[lens < 2] = 1
    first_sub = np.zeros(nvar + 1, dtype=np.int64)
    np.cumsum(nsub, out=first_sub[1:])
    pos = np.zeros(int(first_sub[-1]), dtype=np.int32)
    one = nsub == 1
    pos[first_sub[:-1][one]] = (rng.random(one.sum()) * lens[one]).astype(np.int32)
    two = ~one
    a0 = (rng.random(two.sum()) * (lens[two] - 1)).astype(np.int64)
    a1 = a0 + 1 + (rng.random(two.sum()) * (lens[two] - 1 - a0)).astype(np.int64)
    pos[first_sub[:-1][two]] = a0
    pos[first_sub[:-1][two] + 1] = a1
    code = rng.integers(1, 21, len(pos)).astype(np.uint8)
    wl.append(("c: 200 000 random single and double substitutions over a yeast-sized reference", codes, offs,
               (protein, first_sub, pos, code)))
    return wl


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "variants_bench.json"))
    ap.add_argument("--sample-res", type=float, default=4e8)
    a = ap.parse_args()
    if plaac_b200.lib().plaac_device_count() <= 0:
        sys.exit("variants_bench: no CUDA device")
    info = {"card": card(), "results": []}
    print("card:", info["card"], flush=True)

    for name, c, o, var in workloads():
        r = run_workload(name, c, o, var, a.sample_res)
        info["results"].append(r)
        v, s = r["variant_call"], r["sample"]
        print(f"{name}: {r['variants']} variants, {r['variant_residues']:.3e} residues; variant call "
              f"{v['wall_s_median'] * 1e3:.1f} ms = {v['residues_per_s']:.3e} res/s (H2D {v['h2d_bytes'] / 1e6:.1f} MB, "
              f"D2H {v['d2h_bytes'] / 1e6:.1f} MB); kernels {r['variant_kernels']}; sample {s['residues']:.3e} res: "
              f"device-resident {s['device_resident']['residues_per_s']:.3e} res/s, pinned plaac_score "
              f"{s['host_pinned_plaac_score']['residues_per_s']:.3e} res/s, records equal: {s['records_equal_to_variant_call']}",
              flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(info, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
