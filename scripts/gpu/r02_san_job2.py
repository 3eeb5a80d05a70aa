"""synccheck probe: summary-mode long path on small long proteins (k_long_score alone), then per-residue without records."""
import os, sys
sys.path.insert(0, os.getcwd())
import numpy as np, torch
import plaac_b200
from tests import synth
which = sys.argv[1]
if which == "big": os.environ["PLAAC_LP_BIG_MIN"] = "1024"  # (read when the Scorer is created)
lc, lo = synth.long_proteins(seed=1009, lengths=(1300, 5000, 2049, 9000))
sc = plaac_b200.Scorer(); sc.set_long_path(1024)
if which == "summary":
    s = sc.score(lc, lo)
    print("summary ok", sc.stats().long_proteins)
else:
    dev = torch.device("cuda", 0)
    n = int(lo[-1])
    dc = torch.from_numpy(np.concatenate([lc, np.zeros(64, np.uint8)])).to(dev); do = torch.from_numpy(lo).to(dev)
    u8 = torch.zeros(2 * n, dtype=torch.uint8, device=dev); f64 = torch.zeros(10 * n, dtype=torch.float64, device=dev)
    ptrs = {"vit": u8.data_ptr(), "map": u8.data_ptr() + n}
    for k, nm in enumerate(plaac_b200.RESIDUE_F64): ptrs[nm] = f64.data_ptr() + 8 * k * n
    sc.score_device(dc.data_ptr(), do.data_ptr(), 4, n, 0, residue_ptrs=ptrs, sync=True)
    print("per-residue ok", which, sc.stats().long_proteins)
