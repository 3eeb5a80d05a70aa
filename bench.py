#!/usr/bin/env python
"""bench.py -- residues/s of full PLAAC summary scoring on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path
    python bench.py --impl reference --gpus N ...             # the reference algorithm on the host CPUs
    python bench.py ... --dump-outputs DIR                    # also save a sample of the last step's records

Workload (config.workload): a UniProt-like synthetic proteome (SURVEY.md section 8(d), config 4:
100M proteins / ~35G residues over 8 GPUs), 12.5M proteins per GPU, generated ON DEVICE with
Philox keyed by (seed, global protein index): weak scaling, N=8 is the full config-4 set.
A "step" scores the rank's whole shard once.

  value  : whole-job residues/s with codes+offsets resident in HBM (device-timed, max over ranks)
  e2e    : the same through plaac_score() with pinned HOST buffers (H2D of codes/offsets and D2H of the
           160-byte records inside the timed region)
  roofline: dominant kernel (k_score_summary), CUDA-event time measured inside the library on its stream
  cpu_baseline: the CPU oracle (a line-faithful port of plaac.java; no JVM exists here) on a bounded sample
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "residues/s full PLAAC scoring"
UNIT = "residues/s"
F_PER_AA = 67.0      # SURVEY.md section 8(d): algorithmic fp64 ops per residue, summary mode
B_FIXED_PER_PROT = 168.0  # 160 B record + 8 B offset per protein; + 1 B per residue
SEED = 1004          # config 4
LN_MEDIAN, SIGMA, MIN_LEN, MAX_LEN = math.log(290.0), 0.62, 16, 40000
PRD_RATE, X_RATE = 0.05, 1e-4
# 27 record fields + the protein index in float64, 13 non-finite classes in float32: 55.2 MB at most
DUMP_PROTEINS, DUMP_SEED = 200_000, 0

BG_SCER = [0, 0.0550, 0.0126, 0.0586, 0.0655, 0.0441, 0.0498, 0.0217, 0.0655, 0.0735, 0.0950, 0.0207,
           0.0615, 0.0438, 0.0396, 0.0444, 0.0899, 0.0592, 0.0556, 0.0104, 0.0337, 0]
PRD_28 = [0, 0.04865, 0.00219, 0.01638, 0.00783, 0.02537, 0.07603, 0.0181, 0.02018, 0.01641, 0.02639,
          0.02975, 0.25885, 0.05126, 0.15178, 0.025, 0.10988, 0.03841, 0.01972, 0.00157, 0.05624, 0]


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"must be at least 1, got {v}")
    return v


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--proteins-per-gpu", type=int, default=12_500_000)
    ap.add_argument("--cpu-sample-proteins", type=int, default=0, help="0 = sized automatically")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-multi-ctx", action="store_true",
                    help="skip the single-process multi-GPU side measurement (plaac_score_multi_packed, N > 1 only)")
    ap.add_argument("--no-per-residue", action="store_true", help="skip the config-2 (per-residue mode) side measurement")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the config-5 (long sequences) and ranking side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the records of the last timed step (rank 0's shard, a fixed sample of at most "
                         f"{DUMP_PROTEINS} proteins) as DIR/<field>.npy in float64, with DIR/protein_index.npy; "
                         "NaN and infinities are written as 0 and marked in DIR/<field>_nonfinite.npy")
    return ap.parse_args()


# --------------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def mark(self):
        """Index of the next sample: rows from here on belong to the region that starts now."""
        return len(self.rows)

    def stop(self, first=0, last=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows[first:last]:
            parts = [x.strip() for x in r.split(",")]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "power_w_max": max(power)}


# --------------------------------------------------------------------------------------- CPU arm
def cpu_sample(nprot, seed):
    """Host-side sample of the same distribution (numpy) for the CPU baseline."""
    import numpy as np

    rng = np.random.default_rng(seed)
    lens = np.clip(np.rint(rng.lognormal(LN_MEDIAN, SIGMA, nprot)), MIN_LEN, MAX_LEN).astype(np.int64)
    offsets = np.zeros(nprot + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    bg = np.array(BG_SCER) / sum(BG_SCER)
    codes = rng.choice(22, size=int(offsets[-1]), p=bg).astype(np.uint8)
    codes[rng.random(len(codes)) < X_RATE] = 0
    prd = np.array(PRD_28) / sum(PRD_28)
    for i in np.nonzero(rng.random(nprot) < PRD_RATE)[0]:
        n = int(lens[i])
        seg = int(min(n, rng.integers(60, 301)))
        st = int(rng.integers(0, n - seg + 1))
        codes[offsets[i] + st: offsets[i] + st + seg] = rng.choice(22, size=seg, p=prd)
    return codes, offsets


def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which is not the box's size)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def time_oracle(nprot, nthreads, full_jar_work, repeats=1, keep=None):
    from oracle import orc

    codes, offsets = cpu_sample(nprot, SEED)
    P = orc.make_params()
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        ref = orc.score_batch(P, codes, offsets, full_jar_work=full_jar_work, nthreads=nthreads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    if keep is not None:
        keep.update(codes=codes, offsets=offsets, ref=ref)
    return int(offsets[-1]), best


def check_sample_against_oracle(scorer, kept):
    """The CPU sample the oracle has just scored, through the product path: the oracle as the checker."""
    from oracle import orc
    from tests import parity

    got = scorer.score(kept["codes"], kept["offsets"])
    ref = kept["ref"]
    int_bad = int(sum(int((got[f] != ref[f]).sum()) for f in orc.INT_FIELDS if f != "papa_center"))
    bad = parity.compare_summaries(got, ref, [f for f in orc.INT_FIELDS if f != "papa_center"], orc.DBL_FIELDS)
    cen = int((got["papa_center"] != ref["papa_center"]).sum())
    return {"proteins": int(len(ref)), "int_mismatches": int_bad, "papa_center_differs": cen,
            "max_rel_err": {f: parity.max_rel(got, ref, f) for f in ("llr", "core_score", "hmm_all", "hmm_vit", "papa_combo")},
            "ok": not bad or all(("papa" in b) for b in bad),
            "mismatches": bad[:5],
            "note": "GPU records of the CPU sample vs the oracle's: integers bit-exact, doubles within 1e-9 relative "
                    "(tests/parity.py); a differing PAPA centre is the documented exact-tie class (DESIGN.md 3)"}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU algorithm on the box's host cores.  plaac.jar cannot run
    (no JVM in the image), so this is the oracle port with the jar's dead work switched on, OpenMP over
    proteins on every host thread.  Rank 0 only."""
    if rank != 0:
        return
    from oracle import orc

    nthreads = host_threads()
    nprot = args.cpu_sample_proteins or 3000 * nthreads
    codes, offsets = cpu_sample(nprot, SEED)
    P = orc.make_params()
    nres = int(offsets[-1])
    for _ in range(max(1, min(args.warmup, 1))):
        orc.score_batch(P, codes, offsets, full_jar_work=1, nthreads=nthreads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        orc.score_batch(P, codes, offsets, full_jar_work=1, nthreads=nthreads)
    dt = time.perf_counter() - t0
    value = nres * args.steps / dt
    java = subprocess.run("java -version", shell=True, capture_output=True, text=True)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": nthreads, "kind": "port",
                         "sample": f"{nprot} proteins / {nres} residues of the same synthetic distribution per step; "
                                   "oracle port of plaac.java incl. the jar's dead posterior passes; "
                                   f"JVM {'present' if java.returncode == 0 else 'absent'} (plaac.jar not runnable)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def workload_config(args, world):
    return {"workload": "config4 UniProt-like synthetic proteome shard (lognormal lengths median 290 sigma 0.62, "
                        "yeast background, 5% proteins with injected Q/N-rich segment, X 1e-4), summary mode -c 60 -a 1",
            "proteins_per_gpu": args.proteins_per_gpu, "proteins_total": args.proteins_per_gpu * world,
            "parallelism": f"shard{world} (independent proteins, no collective)",
            "l2": "inputs larger than L2 (shard >> 126 MB); no flush needed"}


# --------------------------------------------------------------------------------------- GPU arm
_JSON_OUT = None


def claim_stdout():
    """stdout carries the one JSON line and nothing else: keep a private handle on it and send everything any library
    prints to fd 1 (NCCL's version banner, for one, at some NCCL_DEBUG settings) to stderr instead."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
    return _JSON_OUT


def emit(line):
    out = claim_stdout()
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    args = parse()
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    # (NCCL_DEBUG is left as the launcher set it: whatever NCCL prints on fd 1 goes to stderr, see claim_stdout)
    import torch
    import torch.distributed as dist

    import plaac_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    L = plaac_b200.lib()
    nprot = args.proteins_per_gpu
    first = rank * nprot

    codes, offsets, ntotal = synth_shard(L, dev, first, nprot)
    summaries = torch.empty(nprot * 160, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()

    scorer = plaac_b200.Scorer(device=local_rank)
    stream = torch.cuda.ExternalStream(scorer.stream(), device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        scorer.score_device(codes.data_ptr(), offsets.data_ptr(), nprot, ntotal, summaries.data_ptr(), sync=True)

    # ---- device-resident timing -------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()  # nvidia-smi needs ~0.1 s to start streaming: started before the warm-up, read for the timed region only
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    m0 = sampler.mark()
    l0 = scorer.stats().kernel_launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    score_ms = []
    ev0.record(stream)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
        score_ms.append(scorer.stats().last_score_ms)
    ev1.record(stream)
    barrier()
    wall = time.perf_counter() - t0
    m1 = sampler.mark()
    clocks = sampler.stop(m0, max(m1, m0 + 1))
    launches = scorer.stats().kernel_launches - l0
    dev_ms = ev0.elapsed_time(ev1)
    t_rank = torch.tensor([dev_ms / 1e3, float(ntotal), wall], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t_rank.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t_rank.clone()
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        t_max, res_total = float(tmax[0]), float(tsum[1])
    else:
        t_max, res_total = float(t_rank[0]), float(ntotal)
    value = res_total * args.steps / t_max
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, summaries, first, nprot)

    # ---- roofline of the dominant kernel (rank-local) ---------------------------------------------
    kern_ms = sum(score_ms) / len(score_ms)
    fp64_peak = C_double()
    L.plaac_bench_fp64_peak(local_rank, 0, fp64_peak.ref(), None)
    peak_ops = fp64_peak.value
    fp64_fma = C_double()
    L.plaac_bench_fp64_peak(local_rank, 1, fp64_fma.ref(), None)
    achieved_ops = F_PER_AA * ntotal / (kern_ms * 1e-3)
    alg_bytes = ntotal + B_FIXED_PER_PROT * nprot
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    # DRAM traffic of the dominant kernel per launch: dram__bytes_read.sum + dram__bytes_write.sum of one
    # `ncu --set full` capture of this command (profiles/traffic.json names the capture and its size); scaled by
    # residues if this run's shard differs from the captured one.
    traffic = None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        traffic = float(tr["dram_bytes"]) * ntotal / float(tr["residues"])
    except Exception:
        pass
    roofline = {
        "bound": "fp64", "kernel": "k_score_summary_v3 (+ k_core_search_jump, same event bracket)",
        "achieved": achieved_ops / 1e12, "peak": peak_ops / 1e12, "unit": "TFLOP/s",
        "frac": achieved_ops / peak_ops, "traffic": traffic,
        "note": "fp64 pipe binds (SURVEY 8d): achieved = 67 algorithmic fp64 ops/residue x residues per launch / "
                "CUDA-event kernel time; peak = DADD issue rate measured by plaac_bench_fp64_peak in this run "
                "(no FMA: the path may not contract a*b+c); DFMA rate for context: %.2f T instr/s" % (fp64_fma.value / 1e12),
        "kernel_ms": kern_ms, "kernel_share_of_step": kern_ms * args.steps / dev_ms,
        "hbm": {"achieved": alg_bytes / (kern_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": alg_bytes / (kern_ms * 1e-3) / 1e9 / hbm_peak,
                "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"},
    }

    # ---- end to end through the public host-buffer call -------------------------------------------
    e2e = None
    e2e_skip = None
    if not args.no_e2e:
        # every rank pins its shard's codes, offsets and records in host memory: make sure the box has room
        need = (ntotal + 8 * (nprot + 1) + 160 * nprot + 4 * (ntotal // 7) + 4 * nprot + 21 * nprot) * max(1, world)
        try:
            with open("/proc/meminfo") as f:
                avail = next(int(x.split()[1]) * 1024 for x in f if x.startswith("MemAvailable"))
        except Exception:
            avail = None
        if avail is not None and need * 1.25 > avail:
            e2e_skip = f"host memory: {need / 1e9:.0f} GB of pinned buffers needed, {avail / 1e9:.0f} GB available"
    if not args.no_e2e and e2e_skip is None:
        e2e = measure_e2e(args, scorer, dev, world, barrier, codes, offsets, summaries, nprot, ntotal, res_total)
    elif e2e_skip is not None:
        e2e = {"value": None, "unit": UNIT, "skipped": e2e_skip}

    # ---- the single-process multi-GPU path (rank 0 drives all N GPUs; the other ranks idle at a host barrier) --------
    multi_ctx = None
    if world > 1 and not args.no_e2e and not args.no_multi_ctx:
        multi_ctx = measure_multi_ctx(args, L, dev, rank, world, nprot)

    # ---- config 2 side measurement: per-residue mode (rank 0, N=1 only) -----------------------------
    per_res = None
    if rank == 0 and world == 1 and not args.no_per_residue:
        per_res = measure_per_residue(L, scorer, dev, hbm_peak)

    # ---- config 5 (long sequences) and on-device ranking side measurements (rank 0, N=1 only) -------
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        extras = measure_extras(scorer, dev, summaries, nprot)

    # ---- CPU baseline (rank 0, N=1 only) -------------------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import orc

        nthreads = host_threads()
        n1 = args.cpu_sample_proteins or 6000
        nres1, dt1 = time_oracle(n1, 1, 1)
        nall = args.cpu_sample_proteins or 3000 * nthreads
        kept = {}
        nresn, dtn = time_oracle(nall, nthreads, 1, keep=kept)
        sample_parity = check_sample_against_oracle(scorer, kept)
        del kept
        nresn2, dtn2 = time_oracle(nall, nthreads, 0)
        cpu = {"value": nresn / dtn, "unit": UNIT, "cores": nthreads, "kind": "port",
               "sample": f"{nall} proteins / {nresn} residues of the same synthetic distribution",
               "single_thread_value": nres1 / dt1,
               "needed_work_only_value": nresn2 / dtn2,
               "gpu_parity_on_sample": sample_parity,
               "note": "oracle/plaac_oracle.c (gcc -O2 -ffp-contract=off), a line-faithful port of plaac.java; "
                       "value includes the posterior passes the jar computes but never prints; "
                       "needed_work_only_value skips them; single_thread_value is the jar's execution model; "
                       "no JVM in the image, plaac.jar itself cannot be timed"}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": t_max / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, world),
            "residues_per_gpu": ntotal, "gpu_launches": int(launches), "clocks": clocks,
            "roofline": roofline, "e2e": e2e, "multi_ctx_e2e": multi_ctx, "cpu_baseline": cpu, "per_residue_mode": per_res,
            "extras": extras,
            "timing": "CUDA events on the library stream around K steps, max over ranks; wall %.3f s" % wall,
        }
        emit(line)
    scorer.close()
    if world > 1:
        dist.destroy_process_group()


def synth_shard(L, dev, first, nprot):
    """Proteins first .. first+nprot-1 of the synthetic proteome, generated on device: (codes, offsets, residues).
    codes carries 64 bytes of padding after the last residue."""
    import numpy as np
    import torch

    lens = torch.empty(nprot, dtype=torch.int64, device=dev)
    rc = L.plaac_bench_synth_lengths(None, SEED, first, nprot, LN_MEDIAN, SIGMA, MIN_LEN, MAX_LEN, lens.data_ptr())
    assert rc == 0
    offsets = torch.zeros(nprot + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=offsets[1:])
    ntotal = int(offsets[-1].item())
    del lens
    codes = torch.empty(ntotal + 64, dtype=torch.uint8, device=dev)
    bg = np.array(BG_SCER, dtype=np.float64)
    prd = np.array(PRD_28, dtype=np.float64)
    rc = L.plaac_bench_synth_residues(None, SEED, first, nprot, offsets.data_ptr(), bg.ctypes.data, prd.ctypes.data,
                                      PRD_RATE, X_RATE, codes.data_ptr())
    assert rc == 0
    return codes, offsets, ntotal


def dump_outputs(out_dir, summaries, first, nprot):
    """The 160-byte records in `summaries` (device) of a fixed, seeded sample of the shard's proteins, one float64 array
    per record field, and the global index of each sampled protein; the same arguments give the same sample.
    Every array written is finite: a record holds NaN where a score is undefined (core_score without a CORE, for one)
    and -Inf as the LLR of a protein shorter than the core, so each double field is written with those entries as 0
    and, beside it,
    <field>_nonfinite (0 finite, 1 NaN, 2 +Inf, 3 -Inf)."""
    import numpy as np
    import torch

    import plaac_b200

    n = min(nprot, DUMP_PROTEINS)
    pick = np.sort(np.random.default_rng(DUMP_SEED).choice(nprot, size=n, replace=False))
    rows = summaries.view(nprot, 160)[torch.from_numpy(pick).to(summaries.device)]
    rec = rows.cpu().numpy().reshape(-1).view(plaac_b200.SUMMARY_DTYPE)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "protein_index.npy"), (first + pick).astype(np.float64))
    for name in plaac_b200.SUMMARY_DTYPE.names:
        v = rec[name].astype(np.float64)
        if rec.dtype[name].kind == "f":
            cls = np.select([np.isnan(v), v == np.inf, v == -np.inf], [1, 2, 3], 0).astype(np.float32)
            np.save(os.path.join(out_dir, name + "_nonfinite.npy"), cls)
            v[cls != 0] = 0.0
        np.save(os.path.join(out_dir, name + ".npy"), v)


def measure_e2e(args, scorer, dev, world, barrier, codes, offsets, summaries, nprot, ntotal, res_total):
    """End to end through the public host-buffer calls, host buffers from plaac_host_alloc (page-locked), H2D of the inputs
    and D2H of the results inside the timed region, wall clock between barriers, max over ranks.  Three transports of the
    SAME scoring (records bit-identical, checked below):
      packed_in_hits_out     plaac_score_packed: radix-22 words (4/7 B per residue) + int32 lengths in, the ranked records
                             of the proteins with a CORE out (what the reference's consumer displays) -- the headline
      packed_in_records_out  the same input, all 160-byte records out
      bytes_in_records_out   plaac_score: 1 B per residue + int64 offsets in, all records out (round 1's figure)"""
    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    import plaac_b200

    L = plaac_b200.lib()
    pb_codes = plaac_b200.PinnedBuffer(ntotal, np.uint8)
    pb_offsets = plaac_b200.PinnedBuffer(nprot + 1, np.int64)
    pb_sum = plaac_b200.PinnedBuffer(nprot * 160, np.uint8)
    nwords = int(L.plaac_packed_words(ntotal))
    pb_words = plaac_b200.PinnedBuffer(max(nwords, 1), np.uint32)
    pb_len = plaac_b200.PinnedBuffer(nprot, np.int32)
    cap = nprot // 8 + 1024          # the synthetic proteome has a CORE in ~5 % of its proteins
    pb_hrec = plaac_b200.PinnedBuffer(cap * 160, np.uint8)
    pb_hidx = plaac_b200.PinnedBuffer(cap, np.int32)
    h_codes, h_offsets, h_sum = (torch.from_numpy(b.array) for b in (pb_codes, pb_offsets, pb_sum))
    h_codes.copy_(codes[:ntotal])
    h_offsets.copy_(offsets)
    torch.cuda.synchronize()
    pb_len.array[:] = np.diff(pb_offsets.array).astype(np.int32)
    t0 = time.perf_counter()
    plaac_b200.pack_words(pb_codes.array, out=pb_words.array)
    pack_s = time.perf_counter() - t0
    hits = plaac_b200.Hits(mode=plaac_b200.HITS_CORE, rank_flags=0, capacity=cap, records=pb_hrec.ptr, index=pb_hidx.ptr,
                           count=0, n_core=0)

    def run_bytes():
        scorer.score_ptr(h_codes.data_ptr(), h_offsets.data_ptr(), nprot, h_sum.data_ptr())

    def run_packed_records():
        scorer._check(L.plaac_score_packed(scorer._h, pb_words.ptr, pb_len.ptr, nprot, ntotal, pb_sum.ptr, None, None))

    def run_packed_hits():
        scorer._check(L.plaac_score_packed(scorer._h, pb_words.ptr, pb_len.ptr, nprot, ntotal, None, None, C.byref(hits)))

    flat = summaries.view(torch.uint8).reshape(-1)

    def records_match():
        # every byte of every record: the host calls score the shard in pipelined chunks, the device call in one piece
        same = True
        piece = 1 << 28
        for lo in range(0, flat.numel(), piece):
            hi = min(flat.numel(), lo + piece)
            same = same and bool(torch.equal(h_sum[lo:hi].to(dev, non_blocking=False), flat[lo:hi]))
        return same

    def hits_match():
        n = int(hits.count)
        rec = summaries.view(torch.float64).view(nprot, 20)
        ncore_dev = int((~torch.isnan(rec[:, 8])).sum().item())
        idx = torch.from_numpy(pb_hidx.array[:n].copy()).to(dev).long()
        got = torch.from_numpy(pb_hrec.array[:n * 160].copy()).to(dev)
        want = summaries.view(torch.uint8).view(nprot, 160)[idx].reshape(-1)
        cs, ll = rec[idx, 8], rec[idx, 7]
        a, b = slice(0, -1), slice(1, None)
        ordered = bool(((cs[a] > cs[b]) | ((cs[a] == cs[b]) & ((ll[a] > ll[b]) | ((ll[a] == ll[b]) & (idx[a] < idx[b]))))).all())
        return {"n_core": int(hits.n_core), "returned": n, "n_core_device_path": ncore_dev,
                "records_equal_device_path": bool(torch.equal(got, want)), "order_verified": ordered,
                "complete": n == int(hits.n_core) == ncore_dev}

    out = {}
    for tag, fn in (("bytes_in_records_out", run_bytes), ("packed_in_records_out", run_packed_records),
                    ("packed_in_hits_out", run_packed_hits)):
        h_sum.zero_()
        for _ in range(2):
            fn()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        barrier()
        dt = time.perf_counter() - t0
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        if tag == "bytes_in_records_out":
            h2d, d2h = ntotal + 8 * (nprot + 1), 160 * nprot
        else:
            h2d = 4 * nwords + 4 * nprot
            d2h = 160 * nprot if tag == "packed_in_records_out" else 164 * int(hits.count)
        bb = torch.tensor([float(h2d), float(d2h)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(bb, op=dist.ReduceOp.SUM)
        v = {"value": res_total * args.steps / float(tt[0]), "unit": UNIT, "ms_per_step": float(tt[0]) / args.steps * 1e3,
             "h2d_bytes_per_step": int(bb[0]), "d2h_bytes_per_step": int(bb[1])}
        if tag == "packed_in_hits_out":
            v["hits"] = hits_match()
        else:
            v["matches_device_path"] = records_match()
            v["records_compared"] = int(nprot)
        out[tag] = v
    head = dict(out["packed_in_hits_out"])
    head["call"] = "plaac_score_packed(words, lengths, hits=PLAAC_HITS_CORE)"
    head["variants"] = {k: out[k] for k in ("packed_in_records_out", "bytes_in_records_out")}
    head["host_pack_s"] = pack_s
    head["note"] = ("host buffers from plaac_host_alloc (page-locked) in every rank (each GPU on its own PCIe link); byte "
                    "counts are whole-job totals counted from the buffers copied; wall clock between barriers, max over "
                    "ranks; packing the residues into radix-22 words is host preprocessing outside the timed region "
                    "(host_pack_s, all host threads), like the FASTA->codes encoding of the one-byte call")
    del h_codes, h_offsets, h_sum
    for b in (pb_codes, pb_offsets, pb_sum, pb_words, pb_len, pb_hrec, pb_hidx):
        b.close()
    return head


def measure_multi_ctx(args, L, dev, rank, world, nprot):
    """The product's multi-GPU path for a host that drives several GPUs from ONE process (a Java or C++ host): rank 0
    holds the shards of all `world` ranks as one batch in page-locked memory (radix-22 words + int32 lengths) and calls
    plaac_score_multi_packed with one ctx per GPU (one host thread each, residue-balanced shards, ranked CORE hits merged on
    the host).  The other ranks wait at a gloo (host) barrier so that their GPUs are idle.  Wall clock around K calls."""
    import ctypes as C

    import numpy as np
    import torch
    import torch.distributed as dist

    import plaac_b200

    host_group = dist.new_group(backend="gloo")
    dist.barrier(group=host_group)
    out = None
    if rank == 0:
        steps = max(2, min(args.steps, 5))
        bg = np.array(BG_SCER, dtype=np.float64)
        prd = np.array(PRD_28, dtype=np.float64)
        ntot_prot = nprot * world
        pb_len = plaac_b200.PinnedBuffer(ntot_prot, np.int32)
        # shard sizes first (lengths are cheap to generate), then one pinned word buffer for the whole batch
        shard_res = []
        for r in range(world):
            lens = torch.empty(nprot, dtype=torch.int64, device=dev)
            L.plaac_bench_synth_lengths(None, SEED, r * nprot, nprot, LN_MEDIAN, SIGMA, MIN_LEN, MAX_LEN, lens.data_ptr())
            pb_len.array[r * nprot:(r + 1) * nprot] = lens.to(torch.int32).cpu().numpy()
            shard_res.append(int(lens.sum().item()))
            del lens
        nres = int(sum(shard_res))
        nwords = int(L.plaac_packed_words(nres))
        pb_words = plaac_b200.PinnedBuffer(nwords, np.uint32)
        pb_tmp = plaac_b200.PinnedBuffer(max(shard_res), np.uint8)
        pos = 0
        t0 = time.perf_counter()
        for r in range(world):
            lens = torch.from_numpy(pb_len.array[r * nprot:(r + 1) * nprot].astype(np.int64)).to(dev)
            offs = torch.zeros(nprot + 1, dtype=torch.int64, device=dev)
            torch.cumsum(lens, 0, out=offs[1:])
            codes = torch.empty(shard_res[r] + 64, dtype=torch.uint8, device=dev)
            L.plaac_bench_synth_residues(None, SEED, r * nprot, nprot, offs.data_ptr(), bg.ctypes.data, prd.ctypes.data,
                                         PRD_RATE, X_RATE, codes.data_ptr())
            torch.from_numpy(pb_tmp.array[:shard_res[r]]).copy_(codes[:shard_res[r]])
            torch.cuda.synchronize()
            pos = plaac_b200.pack_append(pb_tmp.array[:shard_res[r]], pb_words.array, pos)
            del lens, offs, codes
        prep_s = time.perf_counter() - t0
        pb_tmp.close()
        cap = ntot_prot // 8 + 1024
        pb_hrec = plaac_b200.PinnedBuffer(cap * 160, np.uint8)
        pb_hidx = plaac_b200.PinnedBuffer(cap, np.int32)
        hits = plaac_b200.Hits(mode=plaac_b200.HITS_CORE, rank_flags=0, capacity=cap, records=pb_hrec.ptr, index=pb_hidx.ptr,
                               count=0, n_core=0)
        ms = plaac_b200.MultiScorer(devices=list(range(world)))
        handles = (C.c_void_p * world)(*[s._h for s in ms.scorers])

        def run():
            rc = L.plaac_score_multi_packed(handles, world, pb_words.ptr, pb_len.ptr, ntot_prot, nres, None, None, C.byref(hits))
            if rc != 0:
                raise SystemExit("plaac_score_multi_packed failed: %d %s" % (rc, [L.plaac_last_error(s._h) for s in ms.scorers]))

        for _ in range(2):
            run()
        t0 = time.perf_counter()
        for _ in range(steps):
            run()
        dt = time.perf_counter() - t0
        n = int(hits.count)
        rec = np.frombuffer(pb_hrec.array[:n * 160].tobytes(), dtype=plaac_b200.SUMMARY_DTYPE)
        cs, ll, idx = rec["core_score"], rec["llr"], pb_hidx.array[:n].astype(np.int64)
        ordered = bool(np.all((cs[:-1] > cs[1:]) | ((cs[:-1] == cs[1:]) & ((ll[:-1] > ll[1:]) | ((ll[:-1] == ll[1:]) & (idx[:-1] < idx[1:]))))))
        out = {"value": nres * steps / dt, "unit": UNIT, "ms_per_step": dt / steps * 1e3, "steps": steps, "gpus": world,
               "call": "plaac_score_multi_packed(ctxs[0..N), words, lengths, hits=PLAAC_HITS_CORE), one process",
               "proteins": ntot_prot, "residues": nres,
               "h2d_bytes_per_step": 4 * nwords + 4 * ntot_prot, "d2h_bytes_per_step": 164 * n,
               "hits": {"n_core": int(hits.n_core), "returned": n, "order_verified": ordered,
                        "complete": n == int(hits.n_core)},
               "host_prep_s": prep_s,
               "note": "rank 0 alone, every other rank idle at a host barrier; page-locked buffers; wall clock around the calls"}
        ms.close()
        for b in (pb_len, pb_words, pb_hrec, pb_hidx):
            b.close()
    dist.barrier(group=host_group)
    return out


def measure_per_residue(L, scorer, dev, hbm_peak):
    """Config 2 (per-residue table: VIT, MAP, 8 tracks, 2 posteriors = 82 B/residue out), device-resident:
    the yeast-proteome-sized set the config names, and a 200k-protein batch for the bandwidth view."""
    import numpy as np
    import torch

    import plaac_b200

    out = {}
    for tag, nprot in (("yeast_sized_6k", 6000), ("batch_200k", 200000)):
        lens = torch.empty(nprot, dtype=torch.int64, device=dev)
        L.plaac_bench_synth_lengths(None, 1001, 0, nprot, math.log(407.0), 0.66, MIN_LEN, MAX_LEN, lens.data_ptr())
        offsets = torch.zeros(nprot + 1, dtype=torch.int64, device=dev)
        torch.cumsum(lens, 0, out=offsets[1:])
        ntotal = int(offsets[-1].item())
        codes = torch.empty(ntotal + 64, dtype=torch.uint8, device=dev)
        bg = np.array(BG_SCER, dtype=np.float64)
        prd = np.array(PRD_28, dtype=np.float64)
        L.plaac_bench_synth_residues(None, 1001, 0, nprot, offsets.data_ptr(), bg.ctypes.data, prd.ctypes.data, PRD_RATE,
                                     X_RATE, codes.data_ptr())
        u8 = torch.empty(2 * ntotal, dtype=torch.uint8, device=dev)
        stride = (ntotal + 3) & ~3   # track arrays at multiples of 32 bytes (the kernels then use 256-bit stores)
        f64 = torch.empty(10 * stride, dtype=torch.float64, device=dev)
        ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + ntotal}
        for k, nm in enumerate(plaac_b200.RESIDUE_F64):
            ptrs[nm] = f64.data_ptr() + 8 * k * stride
        torch.cuda.synchronize()

        def f():
            scorer.score_device(codes.data_ptr(), offsets.data_ptr(), nprot, ntotal, 0, residue_ptrs=ptrs, sync=True)

        def timed():
            for _ in range(3):
                f()
            ms = []
            for _ in range(5):
                f()
                ms.append(scorer.stats().last_total_ms)
            return sum(ms) / len(ms) * 1e-3

        # long proteins through the per-residue long-sequence path (automatic threshold per batch), and, for contrast,
        # every protein walked by one lane of the bucketed kernels (the round-1 behaviour)
        scorer.set_long_path(-1)
        n0 = scorer.stats().long_proteins
        t = timed()
        nlong = (scorer.stats().long_proteins - n0) // 8
        scorer.set_long_path(0)
        t_walk = timed()
        scorer.set_long_path(8192)
        out[tag] = {"proteins": nprot, "residues": ntotal, "ms": t * 1e3, "residues_per_s": ntotal / t,
                    "hbm_out_gbs": 82.0 * ntotal / t / 1e9, "frac_of_hbm_write_roofline": 83.0 * ntotal / t / 1e9 / hbm_peak,
                    "long_path_proteins": int(nlong), "ms_without_long_path": t_walk * 1e3}
        del u8, f64, codes, offsets, lens
    out["note"] = ("device-resident, CUDA-event time of the whole per-residue pipeline inside the library; 83 algorithmic "
                   "bytes/residue (1 in + 82 out) against the measured HBM peak; automatic long-path threshold "
                   "(plaac_set_long_path(-1)): the longest proteins of the batch go to one thread-block cluster each "
                   "(long_residue.cuh), the rest is latency-bound by the sequential chains of the longest bucket")
    return out


def measure_extras(scorer, dev, summaries, nprot):
    """Config 5: one 35k- and one 100k-residue protein (background composition, three 150-residue Q/N-rich
    segments) alone on the GPU, through the chunked long-sequence path and, for contrast, through the bucketed
    kernel where one lane walks the whole protein.  Ranking: plaac_rank_device over the bench shard's records."""
    import numpy as np
    import torch

    rng = np.random.default_rng(1005)
    bg = np.array(BG_SCER) / sum(BG_SCER)
    prd = np.array(PRD_28) / sum(PRD_28)
    out = {"long_sequences": {}}
    for n in (35000, 100000):
        s = rng.choice(22, size=n, p=bg).astype(np.uint8)
        for frac in (0.10, 0.50, 0.86):
            st = int(n * frac)
            s[st:st + 150] = rng.choice(22, size=150, p=prd)
        d_codes = torch.from_numpy(s).to(dev)
        d_offs = torch.tensor([0, n], dtype=torch.int64, device=dev)
        d_out = torch.zeros(160, dtype=torch.uint8, device=dev)
        torch.cuda.synchronize()
        res = {}
        for tag, min_len in (("long_path_ms", 8192), ("bucketed_kernel_ms", 0)):
            scorer.set_long_path(min_len)
            ms = []
            for it in range(6):
                scorer.score_device(d_codes.data_ptr(), d_offs.data_ptr(), 1, n, d_out.data_ptr(), sync=True)
                if it:
                    ms.append(scorer.stats().last_total_ms)
            res[tag] = sum(ms) / len(ms)
        scorer.set_long_path(8192)
        res["residues_per_s_long_path"] = n / (res["long_path_ms"] * 1e-3)
        # the same protein in per-residue mode (82 B/residue out, no records): cluster path vs single-lane walk
        import plaac_b200
        u8 = torch.empty(2 * n, dtype=torch.uint8, device=dev)
        f64 = torch.empty(10 * n, dtype=torch.float64, device=dev)
        ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + n}
        for k, nm in enumerate(plaac_b200.RESIDUE_F64):
            ptrs[nm] = f64.data_ptr() + 8 * k * n
        d_codes_p = torch.from_numpy(np.concatenate([s, np.zeros(64, np.uint8)])).to(dev)
        for tag, min_len in (("per_residue_long_path_ms", 8192), ("per_residue_single_lane_ms", 0)):
            scorer.set_long_path(min_len)
            ms = []
            for it in range(5):
                scorer.score_device(d_codes_p.data_ptr(), d_offs.data_ptr(), 1, n, 0, residue_ptrs=ptrs, sync=True)
                if it:
                    ms.append(scorer.stats().last_total_ms)
            res[tag] = sum(ms) / len(ms)
        scorer.set_long_path(8192)
        del u8, f64, d_codes_p
        out["long_sequences"]["n%d" % n] = res
    out["long_sequences"]["note"] = ("whole device pipeline of one call (CUDA events inside the library), a single "
                                     "protein on the GPU; both paths give the same 160-byte record bit for bit, and the same per-residue "
                                     "arrays bit for bit (per_residue_*: posteriors, MAP and Viterbi parse, eight tracks)")
    out["fasta_ingest"] = measure_ingest(scorer, dev)
    order = torch.empty(nprot, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    ts = []
    for it in range(3):
        t0 = time.perf_counter()
        ncore = scorer.rank_device(summaries.data_ptr(), nprot, order.data_ptr())
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    # the order is checked where it lies: COREscore desc, then LLR desc, then input index asc; no-CORE rows last
    rec = summaries.view(torch.float64).view(nprot, 20)   # 160 B = 20 x 8 B; doubles start at byte 56: llr, core_score
    idx = order.long()
    cs, ll = rec[idx, 8], rec[idx, 7]

    def in_order(p, s, i):
        a, b = slice(0, -1), slice(1, None)
        return bool(((p[a] > p[b]) | ((p[a] == p[b]) & ((s[a] > s[b]) | ((s[a] == s[b]) & (i[a] < i[b]))))).all())

    ok = (not bool(torch.isnan(cs[:ncore]).any())) and bool(torch.isnan(cs[ncore:]).all())
    ok = ok and in_order(cs[:ncore], ll[:ncore], idx[:ncore])
    ok = ok and in_order(torch.zeros_like(ll[ncore:]), ll[ncore:], idx[ncore:])
    ok = ok and bool((torch.sort(idx).values == torch.arange(nprot, device=dev)).all())
    del rec, idx, cs, ll
    out["ranking"] = {"records": nprot, "with_core": ncore, "ms": min(ts) * 1e3, "order_verified": ok,
                      "note": "plaac_rank_device: COREscore desc, LLR desc, no-CORE rows last (web/lib/server.rb:222-229); "
                              "wall clock around the call (it ends with a stream synchronise)"}
    return out


def measure_ingest(scorer, dev):
    """Row N2: raw FASTA text (60-column lines, '>' names) already in HBM -> residue codes, offsets, name spans and the
    22-bin background counts (plaac_ingest_fasta_device).  Text of 300 k synthetic proteins (~130 MB)."""
    import ctypes as C

    import numpy as np
    import torch

    import plaac_b200

    rng = np.random.default_rng(7)
    nrec = 300000
    lens = np.clip(np.rint(rng.lognormal(LN_MEDIAN, SIGMA, nrec)), MIN_LEN, MAX_LEN).astype(np.int64)
    ntot = int(lens.sum())
    bg = np.array(BG_SCER) / sum(BG_SCER)
    letters = np.frombuffer(b"XACDEFGHIKLMNPQRSTVWY*", dtype=np.uint8)
    res = letters[rng.choice(22, size=ntot, p=bg)]
    # text layout: ">p<i>\n" then the sequence in lines of 60
    starts = np.concatenate([[0], np.cumsum(lens)])
    parts = []
    for i in range(nrec):
        parts.append(b">p%d\n" % i)
        s = res[starts[i]:starts[i + 1]]
        nl = (len(s) + 59) // 60
        buf = np.full(len(s) + nl, 10, dtype=np.uint8)
        idx = np.arange(len(s))
        buf[idx + idx // 60] = s
        parts.append(buf.tobytes())
    text = b"".join(parts)
    nbytes = len(text)
    d_text = torch.frombuffer(bytearray(text), dtype=torch.uint8).to(dev)
    d_codes = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d_offs = torch.empty(nrec + 2, dtype=torch.int64, device=dev)
    d_npos = torch.empty(nrec + 1, dtype=torch.int64, device=dev)
    d_nlen = torch.empty(nrec + 1, dtype=torch.int32, device=dev)
    d_flags = torch.zeros(nrec + 8, dtype=torch.uint8, device=dev)
    d_bg = torch.zeros(22, dtype=torch.int64, device=dev)
    idx = plaac_b200.capi.FastaIndex()
    L = plaac_b200.lib()
    torch.cuda.synchronize()
    ts = []
    for it in range(4):
        t0 = time.perf_counter()
        rc = L.plaac_ingest_fasta_device(scorer._h, d_text.data_ptr(), nbytes, d_codes.data_ptr(), d_offs.data_ptr(),
                                         d_npos.data_ptr(), d_nlen.data_ptr(), d_flags.data_ptr(), nrec + 1, C.byref(idx),
                                         d_bg.data_ptr())
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
        assert rc == 0 and idx.nrec == nrec and idx.nres == ntot, (rc, idx.nrec, idx.nres)
    t = min(ts[1:])
    return {"text_bytes": nbytes, "records": nrec, "residues": ntot, "ms": t * 1e3, "text_gb_per_s": nbytes / t / 1e9,
            "note": "plaac_ingest_fasta_device (5 kernels + background histogram), text resident in HBM; wall clock around "
                    "the call, which ends with a stream synchronise"}


class C_double:
    def __init__(self):
        import ctypes

        self._c = ctypes.c_double(0.0)
        self._ctypes = ctypes

    def ref(self):
        return self._ctypes.byref(self._c)

    @property
    def value(self):
        return float(self._c.value)


if __name__ == "__main__":
    main()
