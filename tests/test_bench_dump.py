"""bench.py --dump-outputs: the arrays it writes are the records the timed path computed, for a fixed sample of proteins."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import plaac_b200

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_records_of_the_timed_path(tmp_path):
    import torch

    import bench

    nprot = bench.DUMP_PROTEINS + 50_000   # larger than the sample: the dump is a subset
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                        "--proteins-per-gpu", str(nprot), "--no-e2e", "--no-cpu-baseline", "--no-per-residue",
                        "--no-extras", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2

    fields = plaac_b200.SUMMARY_DTYPE.names
    doubles = [n for n in fields if plaac_b200.SUMMARY_DTYPE[n].kind == "f"]
    names = ("protein_index",) + fields + tuple(n + "_nonfinite" for n in doubles)
    assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in names)
    got = {n: np.load(out / (n + ".npy")) for n in names}
    for n, a in got.items():
        assert a.dtype in (np.float32, np.float64) and a.shape == (bench.DUMP_PROTEINS,), n
        assert np.isfinite(a).all(), n
    assert sum(os.path.getsize(out / (n + ".npy")) for n in names) <= 64_000_000
    idx = got["protein_index"].astype(np.int64)
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < nprot

    # the same shard scored directly through the device-resident call
    dev = torch.device("cuda", 0)
    codes, offsets, ntotal = bench.synth_shard(plaac_b200.lib(), dev, 0, nprot)
    recs = torch.empty(nprot * 160, dtype=torch.uint8, device=dev)
    sc = plaac_b200.Scorer(device=0)
    sc.score_device(codes.data_ptr(), offsets.data_ptr(), nprot, ntotal, recs.data_ptr(), sync=True)
    sc.close()
    want = recs.cpu().numpy().view(plaac_b200.SUMMARY_DTYPE)[idx]
    for n in fields:
        w = want[n].astype(np.float64)
        if n in doubles:
            cls = got[n + "_nonfinite"]
            assert (cls == np.select([np.isnan(w), w == np.inf, w == -np.inf], [1, 2, 3], 0)).all(), n
            assert (got[n][cls != 0] == 0).all(), n
            w = np.where(cls == 0, w, 0.0)
        assert (got[n] == w).all(), n
    # proteins without a CORE are in the sample: the NaN path is exercised
    assert (got["core_score_nonfinite"] == 1).any() and (got["core_score_nonfinite"] == 0).any()
