"""Per-residue mode timings: yeast-sized 6k set and 200k batch per long-path threshold; single long proteins."""
import json, math, os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
import plaac_b200, bench
L = plaac_b200.lib(); dev = torch.device("cuda", 0)
sc = plaac_b200.Scorer()
out = {}

def bufs(ntotal):
    u8 = torch.empty(2 * ntotal, dtype=torch.uint8, device=dev)
    stride = (ntotal + 3) & ~3
    f64 = torch.empty(10 * stride, dtype=torch.float64, device=dev)
    ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + ntotal}
    for k, nm in enumerate(plaac_b200.RESIDUE_F64):
        ptrs[nm] = f64.data_ptr() + 8 * k * stride
    return u8, f64, ptrs

def timeit(codes, offsets, nprot, ntotal, ptrs, reps=5):
    ms = []
    for it in range(reps + 2):
        sc.score_device(codes.data_ptr(), offsets.data_ptr(), nprot, ntotal, 0, residue_ptrs=ptrs, sync=True)
        if it >= 2: ms.append(sc.stats().last_total_ms)
    return sum(ms) / len(ms)

sets = [("yeast_sized_6k", 6000), ("batch_200k", 200000)]
if len(sys.argv) > 1 and sys.argv[1] == "small": sets = sets[:1]
for tag, nprot in sets:
    lens = torch.empty(nprot, dtype=torch.int64, device=dev)
    L.plaac_bench_synth_lengths(None, 1001, 0, nprot, math.log(407.0), 0.66, bench.MIN_LEN, bench.MAX_LEN, lens.data_ptr())
    offsets = torch.zeros(nprot + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lens, 0, out=offsets[1:])
    ntotal = int(offsets[-1].item())
    codes = torch.empty(ntotal + 64, dtype=torch.uint8, device=dev)
    bg = np.array(bench.BG_SCER, dtype=np.float64); prd = np.array(bench.PRD_28, dtype=np.float64)
    L.plaac_bench_synth_residues(None, 1001, 0, nprot, offsets.data_ptr(), bg.ctypes.data, prd.ctypes.data, bench.PRD_RATE, bench.X_RATE, codes.data_ptr())
    u8, f64, ptrs = bufs(ntotal)
    res = {"residues": ntotal, "max_len": int(lens.max().item())}
    for thr in (0, 8192, -1, 1024, 2048, 4096):
        sc.set_long_path(thr)
        n0 = sc.stats().long_proteins
        ms = timeit(codes, offsets, nprot, ntotal, ptrs)
        res["thr_%d" % thr] = {"ms": ms, "long_per_call": (sc.stats().long_proteins - n0) // 7}
        print(tag, thr, res["thr_%d" % thr], flush=True)
    out[tag] = res
    del u8, f64, codes, offsets, lens

rng = np.random.default_rng(1005)
for n in (9000, 35000, 100000):
    s = rng.choice(22, size=n, p=np.array(bench.BG_SCER) / np.sum(bench.BG_SCER)).astype(np.uint8)
    for frac in (0.10, 0.50, 0.86):
        st = int(n * frac); s[st:st + 150] = rng.choice(22, size=150, p=np.array(bench.PRD_28) / np.sum(bench.PRD_28))
    codes = torch.from_numpy(np.concatenate([s, np.zeros(64, np.uint8)])).to(dev)
    offsets = torch.tensor([0, n], dtype=torch.int64, device=dev)
    u8, f64, ptrs = bufs(n)
    res = {}
    for tag, thr, env in (("long_path", 1024, {}), ("long_path_one_cta", 1024, {"PLAAC_LP_BIG_MIN": "10000000"}), ("cluster8", 1024, {"PLAAC_LP_BIG_MIN": "1024"}), ("single_lane_walk", 0, {})):
        for k, v in env.items(): os.environ[k] = v
        sc = plaac_b200.Scorer()  # (PLAAC_LP_BIG_MIN is read when a Scorer is created)
        sc.set_long_path(thr)
        res[tag + "_ms"] = timeit(codes, offsets, 1, n, ptrs)
        sc.close()
        for k in env: del os.environ[k]
    print(n, res, flush=True)
    out["n%d" % n] = res
os.makedirs("gpurun_out", exist_ok=True)
json.dump(out, open("gpurun_out/r02_resmode.json", "w"), indent=1)
