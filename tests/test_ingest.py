"""GPU FASTA ingest (N2) and background counts (N3) against a Python restatement of the jar's reader
(fastareader plaac.java:4302-4375, string2aa :1764, '*' strip :758, computeaafreq/isvalidprotein :1655-1739)."""
import re
import subprocess

import numpy as np
import pytest

import plaac_b200
from oracle import orc
from plaac_b200 import build as pb

pytestmark = pytest.mark.gpu


def java_readlines(data: bytes):
    """BufferedReader.readLine: \\n, \\r or \\r\\n end a line; no empty line after a final terminator."""
    lines = re.split(rb"\r\n|\n|\r", data)
    if lines and lines[-1] == b"":
        lines.pop()
    return lines


def reference_reader(data: bytes):
    """(name, unstripped sequence bytes, trimmed?) per record, exactly as the jar iterates them."""
    recs = []
    lines = java_readlines(data)
    i, ondeck, name, trimmed = 0, False, None, False
    while True:
        if not ondeck:  # hasmorefastas: skip to the next '>' line; the name is trimmed
            while i < len(lines) and not (len(lines[i]) > 0 and lines[i][:1] == b">"):
                i += 1
            if i >= len(lines):
                break
            name, trimmed = lines[i].strip(bytes(range(33)))[1:], True
            i += 1
        seq = b""
        ondeck = False
        nxt = None
        while i < len(lines):  # nextfasta
            ln = lines[i]
            i += 1
            if len(ln) == 0:
                break
            if ln[:1] == b">":
                ondeck, nxt = True, ln[1:]
                break
            seq += ln
        recs.append((name.decode("latin-1"), seq, trimmed))
        if ondeck:
            name, trimmed = nxt, False
    return recs


def expected(data: bytes):
    recs = reference_reader(data)
    seqs = [orc.encode(s, strip_stop=True) if len(s) else np.zeros(0, np.uint8) for _, s, _ in recs]
    codes, offs = orc.pack(seqs) if seqs else (np.zeros(0, np.uint8), np.zeros(1, np.int64))
    counts = np.zeros(22)
    for _, s, _ in recs:
        aa = orc.encode(s, strip_stop=False) if len(s) else np.zeros(0, np.uint8)
        m = len(aa)
        if m == 0:
            continue
        valid = aa[m - 1] != 0 and not any(aa[i] in (0, 21) for i in range(1, m - 1))
        if valid:
            counts += np.bincount(aa, minlength=22)
    return [n for n, _, _ in recs], codes, offs, counts


CASES = {
    "plain": b">a\nMKV\nAC\n>b desc text \nQQNN*\n",
    "crlf_and_cr": b">a x\r\nMKV\r\nAC*\r\n>b\rQN\rNQ\r>c\r\n\r\n>d\nAA\n",
    "blank_ends_record": b"junk before\n>a\nMK\n\nIGNORED LINE\nalso ignored\n>b  \nQQ\n\n\n>c\nNN",
    "untrimmed_lines": b">a\n M K V \n\tAC1\n>b\nmkv*acd\n*\n",
    "stars": b">a\n*\n>b\n**\n>c\nAB*\nCD\n>d\nAB*\n\nCD\n>e\nAB* \n>f\nA*B*",
    "empty_records": b">a\n>b\n>c\n\n>d\nMM\n>e",
    "no_trailing_newline": b">only\nMKVQQNNQQ",
    "no_records": b"just text\nno header\n",
    "empty": b"",
    "header_like_inside": b">a\nMK>V\n>b>c\nQ\n",
    "x_and_invalid": b">v1\nMKVA\n>bad_inner_x\nMXKA\n>bad_last_x\nMKAX\n>first_x_ok\nXKVA\n>star_inside\nMK*VA\n>star_end\nMKVA*\n>single\nX\n",
}


@pytest.fixture(scope="module")
def scorer():
    s = plaac_b200.Scorer()
    yield s
    s.close()


@pytest.mark.parametrize("name", sorted(CASES))
def test_ingest_semantics(scorer, name):
    data = CASES[name]
    got = scorer.ingest_fasta(data, bg_counts=True)
    names, codes, offs, counts = expected(data)
    assert got["names"] == names
    assert got["offsets"].tolist() == offs.tolist()
    assert got["codes"].tolist() == codes.tolist()
    assert got["bg_counts"].tolist() == counts.tolist()


def test_ingest_large_random_and_scoring_equivalence(scorer):
    """Random FASTA with every quirk, larger than many 4 KB tiles; the ingested arrays score identically to the
    host-encoded ones; tile boundaries fall everywhere because lines have random lengths."""
    rng = np.random.default_rng(42)
    alphabet = np.frombuffer(b"ACDEFGHIKLMNPQRSTVWYacdxXBZ* 1", dtype=np.uint8)
    parts = []
    for r in range(3000):
        parts.append(b">rec%d some text%s" % (r, b"  " if r % 7 == 0 else b""))
        term = [b"\n", b"\r\n", b"\r"][r % 3]
        parts.append(term)
        n = int(rng.integers(0, 900))
        seq = alphabet[rng.integers(0, len(alphabet) - (0 if r % 5 == 0 else 3), n)].tobytes()
        if r % 4 == 0:
            seq += b"*"
        w = int(rng.integers(1, 120))
        for k in range(0, len(seq), w):
            parts.append(seq[k:k + w] + term)
        if r % 11 == 0:
            parts.append(term + b"skipped text" + term)
    data = b"".join(parts)
    assert len(data) > 1_000_000
    got = scorer.ingest_fasta(data, bg_counts=True)
    names, codes, offs, counts = expected(data)
    assert got["names"] == names
    assert got["offsets"].tolist() == offs.tolist()
    assert (got["codes"] == codes).all()
    assert got["bg_counts"].tolist() == counts.tolist()
    a = scorer.score(got["codes"], got["offsets"])
    b = scorer.score(codes, offs)
    assert a.tobytes() == b.tobytes()


def test_ingest_matches_host_cli_background_counts(scorer, tmp_path):
    """-b count mode of the C++ host (its own reader) == GPU ingest + k_bg_hist."""
    pb.build_lib()
    cli = pb.build_cli()
    data = CASES["x_and_invalid"] + CASES["crlf_and_cr"] + b"\n" + CASES["stars"]
    fa = tmp_path / "x.fa"
    fa.write_bytes(data)
    out = subprocess.run([cli, "-b", str(fa)], capture_output=True, text=True).stdout
    cli_counts = [float(l.split(" # ")[0]) for l in out.strip().split("\n")]
    got = scorer.ingest_fasta(data, bg_counts=True)
    assert got["bg_counts"].tolist() == cli_counts

