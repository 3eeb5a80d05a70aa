"""Parity against the REFERENCE ITSELF: web/bin/plaac.jar's bytecode, executed by tests/golden/minijvm.py (no JVM
exists in this image), on the reference's own example proteins and on edge cases.  The oracle must reproduce every
number the jar prints BIT FOR BIT (same operation order, same libm behind Math.log/exp); the CUDA path must match
within the tolerance classes of tests/parity.py."""
import math

import numpy as np
import pytest

from oracle import orc
from tests import jarvec, parity


@pytest.mark.parametrize("which", ["prions_summary", "edge_summary", "edge_alt_summary", "long_summary", "human_summary", "human_F_summary", "human_b_summary"])
def test_oracle_summary_is_bit_identical_to_the_jar(which):
    enc, kw, rows = jarvec.scenario(which)
    codes, offs = orc.pack([c for _, c in enc])
    ref = orc.score_batch(orc.make_params(**kw), codes, offs)
    for (name, aa), r, row in zip(enc, ref, rows):
        assert row["SEQid"] == name
        for k, e in jarvec.expected_cells(r).items():
            g = jarvec.val(row[k])
            if isinstance(e, float):
                assert (math.isnan(e) and math.isnan(g)) or e == g, (name, k, e, g)
            else:
                assert e == g, (name, k, e, g)
        # string columns: COREaa, STARTaa, ENDaa, PRDaa, PAPAaa (:915-945)
        names = orc.AANAMES

        def sub(r1, r2):
            m = len(aa)
            r1 = max(r1, 0)
            r2 = max(r2, r1)
            r1, r2 = min(r1, m - 1), min(r2, m - 1)
            return "".join(names[c] for c in aa[r1:r2 + 1])

        if r["prd_end"] - r["prd_start"] + 1 >= kw.get("core_len", 60):
            want = [sub(r["core_start"], r["core_end"]), sub(r["prd_start"], r["prd_start"] + 14),
                    sub(r["prd_end"] - 14, r["prd_end"]), sub(r["prd_start"], r["prd_end"])]
        else:
            want = ["-"] * 4
        assert [row["COREaa"], row["STARTaa"], row["ENDaa"], row["PRDaa"]] == want, name
        hw = kw.get("ww2", 41) // 2  # :944 submatrix(aa, papamaxcenter - ww2/2, papamaxcenter + ww2/2)
        assert row["PAPAaa"] == sub(r["papa_center"] - hw, r["papa_center"] + hw), name


@pytest.mark.parametrize("which", ["prions_residue", "edge_residue", "edge_alt_residue", "long_residue"])
def test_oracle_per_residue_is_bit_identical_to_the_jar(which):
    enc, kw, prots = jarvec.scenario(which)
    P = orc.make_params(**kw)
    for (name, aa), pr in zip(enc, prots):
        c, o = orc.pack([aa])
        tr = orc.residue_batch(P, c, o)
        assert pr["aa"] == "".join(orc.AANAMES[x] for x in aa)
        assert tr["vit"].tolist() == pr["vit"], name
        assert tr["map"].tolist() == pr["map"], name
        for k, ok in jarvec.RES_MAP.items():
            g = np.array([jarvec.val(v) for v in pr[k]])
            assert (np.isnan(g) == np.isnan(tr[ok])).all(), (name, k)
            m = ~np.isnan(g)
            assert (g[m] == tr[ok][m]).all(), (name, k)
        g = np.array([[jarvec.val(v) for v in p2] for p2 in pr["post"]])
        assert (g[:, 0] == tr["post_bg"]).all() and (g[:, 1] == tr["post_prd"]).all(), name


def test_parameter_block_matches_the_jar():
    """fg/bg/llr as the jar prints them (## lines, %.5f) == the oracle's parameter chain."""
    J = jarvec.load()
    from tests.test_host_cli import java_fmt

    for tag, sc in (("prions_params", "prions_summary"), ("edge_params", "edge_summary"), ("human_params", "human_summary"),
                    ("edge_alt_params", "edge_alt_summary"), ("human_F_params", "human_F_summary"),
                    ("human_b_params", "human_b_summary")):
        _, kw, _ = jarvec.scenario(sc)
        P = orc.make_params(**kw)
        for key, vec in (("fg_used", P.fg), ("bg_scer", P.bgscer), ("bg_input", P.bgthis), ("bg_used", P.bg), ("plaac_llr", P.llr),
                         ("papa_lods", P.papa_lod)):
            want = "## " + key + ": {" + "".join(f"{n}={java_fmt(v, 5)};" for n, v in zip(orc.AANAMES, vec)) + "}"
            assert J[tag][key] == want, (tag, key)


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prions_summary", "edge_summary", "edge_alt_summary", "long_summary", "long_summary_bucketed",
                                   "human_summary", "human_F_summary", "human_b_summary"])
def test_cuda_summary_against_the_jar(which):
    """long_summary: 4 500 and 9 000 residues, scored by the chunked long-sequence path (scan of max-plus chunk
    matrices, warm-started forward chunks, binade-frame second pass) and, `_bucketed`, by the bucketed kernel:
    both against the numbers the jar's own bytecode produced."""
    import plaac_b200

    bucketed = which.endswith("_bucketed")
    enc, kw, rows = jarvec.scenario(which.replace("_bucketed", ""))
    codes, offs = plaac_b200.pack([c for _, c in enc])
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    sc.set_long_path(0 if bucketed else 4096)
    got = sc.score(codes, offs)
    if which.startswith("long"):
        assert sc.stats().long_proteins == (0 if bucketed else 2)
    sc.close()
    exact = ("LLR", "NLLR", "COREscore", "PRDscore", "HMMall", "HMMvit", "FImeanhydro", "FImeancharge", "FImeancombo")
    nties = 0
    for (name, aa), r, row in zip(enc, got, rows):
        cells = jarvec.expected_cells(r)
        cen_same = cells["PAPAcen"] == jarvec.val(row["PAPAcen"])
        nties += not cen_same
        for k, e in cells.items():
            g = jarvec.val(row[k])
            if k.startswith("PAPA") and not cen_same:
                continue  # documented exact-tie class (plateaus); covered against the oracle in test_gpu_parity
            if isinstance(e, float):
                if k in exact:  # reference-order columns
                    assert (math.isnan(e) and math.isnan(g)) or abs(e - g) <= 1e-13 * max(abs(g), 1.0), (name, k, e, g)
                else:
                    assert bool(parity.close(e, g, 0.1)), (name, k, e, g)
            else:
                assert e == g, (name, k, e, g)
    assert nties <= 3, nties


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["prions_residue", "edge_residue", "edge_alt_residue", "long_residue", "long_residue_cluster"])
def test_cuda_per_residue_against_the_jar(which, monkeypatch):
    """long_residue: the 4 500- and 9 000-residue proteins through the per-residue long-sequence path (k_long_post; one
    CTA per protein, and with `_cluster` a cluster of eight) against the jar's own per-residue table."""
    import plaac_b200

    cluster = which.endswith("_cluster")
    which = which.replace("_cluster", "")
    enc, kw, prots = jarvec.scenario(which)
    codes, offs = plaac_b200.pack([c for _, c in enc])
    if cluster:
        monkeypatch.setenv("PLAAC_LP_BIG_MIN", "1024")  # (read when the Scorer is created)
    sc = plaac_b200.Scorer(plaac_b200.default_params(**kw))
    if which == "long_residue":
        sc.set_long_path(1024)
    _, res = sc.score(codes, offs, per_residue=True)
    if which == "long_residue":
        assert sc.stats().long_proteins == 2
    sc.close()
    for i, ((name, aa), pr) in enumerate(zip(enc, prots)):
        lo, hi = int(offs[i]), int(offs[i + 1])
        assert res["vit"][lo:hi].tolist() == pr["vit"], name
        assert res["map"][lo:hi].tolist() == pr["map"], name
        for k, ok in jarvec.RES_MAP.items():
            g = np.array([jarvec.val(v) for v in pr[k]])
            assert (np.isnan(g) == np.isnan(res[ok][lo:hi])).all(), (name, k)
            assert parity.close(res[ok][lo:hi], g, parity.SCALE[ok]).all(), (name, k)
        g = np.array([[jarvec.val(v) for v in p2] for p2 in pr["post"]])
        assert parity.close(res["post_bg"][lo:hi], g[:, 0], 1.0).all(), name
        assert parity.close(res["post_prd"][lo:hi], g[:, 1], 1.0).all(), name
