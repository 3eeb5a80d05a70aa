"""Small long-sequence per-residue job for compute-sanitizer: both cluster classes, with and without records, lean call."""
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
import plaac_b200
from tests import synth
from oracle import orc
lc, lo = synth.long_proteins(seed=1009, lengths=(1300, 5000, 2049, 9000))
sc_, so = synth.proteome(60, seed=5, median=300.0)
codes = np.concatenate([sc_, lc]); lens = np.concatenate([np.diff(so), np.diff(lo)])
offs = np.zeros(len(lens) + 1, np.int64); np.cumsum(lens, out=offs[1:])
sc = plaac_b200.Scorer(); sc.set_long_path(1024)
ref_s = orc.score_batch(orc.make_params(), codes, offs)
got_s = sc.score(codes, offs)   # records only: k_long_post (forward + Viterbi) beside k_long_score, k_long_final, k_long_fix
for f in ("core_start", "core_end", "vit_maxrun", "llr_start", "mw_score", "fi_numaa"):
    assert (got_s[f] == ref_s[f]).all(), f
assert np.abs(got_s["hmm_all"] - ref_s["hmm_all"]).max() < 1e-9 and np.abs(got_s["hmm_vit"] - ref_s["hmm_vit"]).max() < 1e-9
for big in (None, "1024"):
    if big:
        os.environ["PLAAC_LP_BIG_MIN"] = big  # (read when a Scorer is created)
        sc = plaac_b200.Scorer(); sc.set_long_path(1024)
    summ, res = sc.score(codes, offs, per_residue=True)
    dev = torch.device("cuda", 0)
    dc = torch.from_numpy(np.concatenate([codes, np.zeros(64, np.uint8)])).to(dev); do = torch.from_numpy(offs).to(dev)
    n = int(offs[-1])
    u8 = torch.zeros(2 * n, dtype=torch.uint8, device=dev); f64 = torch.zeros(10 * n, dtype=torch.float64, device=dev)
    ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + n}
    for k, nm in enumerate(plaac_b200.RESIDUE_F64): ptrs[nm] = f64.data_ptr() + 8 * k * n
    sc.score_device(dc.data_ptr(), do.data_ptr(), len(lens), n, 0, residue_ptrs=ptrs, sync=True)
    h8 = u8.cpu().numpy()
    assert (h8[:n] == res["vit"]).all() and (h8[n:] == res["map"]).all()
    assert (f64.cpu().numpy()[8 * n:9 * n] == res["post_bg"]).all()
ref = orc.residue_batch(orc.make_params(), codes, offs)
assert (ref["vit"] == res["vit"]).all() and (ref["map"] == res["map"]).all()
assert np.abs(ref["post_prd"] - res["post_prd"]).max() < 1e-9
print("san job ok", sc.stats().long_proteins)
