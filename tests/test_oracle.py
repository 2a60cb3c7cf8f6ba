"""CPU tests of the oracle: the plain-C restatement (oracle/bin/crumble_oracle) against the
golden vectors generated from the verbatim reference build (oracle/_ref), against oracle/_ref
itself when it is present, and against the reference's own known answers (SURVEY.md §9.5)."""
import hashlib
import json
import os
import struct
import subprocess
import tempfile
from pathlib import Path

import numpy as np
import pytest

import crumble_b200 as cb
from util import PORT_BIN, REF_BIN, ROOT, run_oracle, valid_mask

GOLD = json.load(open(ROOT / "tests" / "golden" / "golden.json"))
GDIR = ROOT / "tests" / "golden"
EDGE = {"l9": ["-9"], "l1B": ["-1", "-B"], "l5q30": ["-5", "-q30"], "l3U35": ["-3", "-U35", "-Y0.2"],
        "l9r": ["-9", "-r", "chrA:900-1600"], "l1r": ["-1", "-r", "chrA:1200-2100"]}


def sim(name):
    g = GOLD[name]
    data, nr, nb = cb.simulate(g["preset"], g["scale"], g["seed"], threads=2)
    assert hashlib.sha256(data.tobytes()).hexdigest() == g["input_sha256"], "synthetic generator is not reproducible"
    return data


@pytest.mark.parametrize("name", sorted(GOLD))
def test_port_matches_golden(name):
    data = sim(name)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish()
    m = valid_mask(bb)
    for args, exp in GOLD[name]["runs"].items():
        r = run_oracle(data, args.split(), binary=PORT_BIN, kind="port")
        assert hashlib.sha256(r["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"], args
        assert r["bed"] == exp["bed"], args
        assert r["counters"] == exp["counters"], args


@pytest.mark.skipif(not REF_BIN.exists(), reason="oracle/_ref not built (make -C oracle ref REF=<crumble source tree>)")
def test_port_matches_reference_binary_fresh_seed():
    data, _, _ = cb.simulate("C1", 0.05, 777, threads=2)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish()
    m = valid_mask(bb)
    for args in (["-9"], ["-1", "-B"], ["-3"]):
        a = run_oracle(data, args, binary=PORT_BIN, kind="port")
        b = run_oracle(data, args, binary=REF_BIN, kind="reference")
        assert np.array_equal(a["qual"][m], b["qual"][m]) and a["bed"] == b["bed"] and a["counters"] == b["counters"]


def run_cli_sam(binary, args, sam_in, env_extra=None):
    with tempfile.TemporaryDirectory() as td:
        out, bed = os.path.join(td, "o.sam"), os.path.join(td, "o.bed")
        subprocess.run([str(binary), "-z"] + args + ["-b", bed, str(sam_in), out], check=True, stderr=subprocess.DEVNULL, stdout=subprocess.DEVNULL,
                       env=dict(os.environ, **(env_extra or {})))
        quals = [(l.rstrip("\n").split("\t")[0], l.rstrip("\n").split("\t")[10]) for l in open(out) if not l.startswith("@")]
        return quals, open(bed).read()


@pytest.mark.parametrize("tag", sorted(EDGE))
def test_port_edge_cases(tag):
    """odd CIGARs (leading/trailing S and I, D, N, P, =/X, adjacent D+I), '*' sequences, FUNMAP-placed and
    unplaced reads, qualities above the cap, a 600 bp read, STR indels, clip pile-up, region iteration."""
    quals, bed = run_cli_sam(PORT_BIN, EDGE[tag], GDIR / "edge_cases.sam")
    exp = [tuple(l.rstrip("\n").split("\t")) for l in open(GDIR / f"edge_cases.{tag}.qual.txt")]
    assert quals == exp
    assert bed == open(GDIR / f"edge_cases.{tag}.bed").read()


def column_dump(args, data):
    with tempfile.TemporaryDirectory() as td:
        fin, dump = os.path.join(td, "i.ubam"), os.path.join(td, "cols.bin")
        data.tofile(fin)
        env = dict(os.environ); env["ORACLE_COLUMN_DUMP"] = dump
        subprocess.run([str(PORT_BIN), "-z"] + args + [fin, "mem:x"], check=True, env=env)
        return np.fromfile(dump, dtype=cb.api.COLUMN_DTYPE)


def test_port_columns_match_reference_debug_dump():
    """per-column call and score against the reference's own -DDEBUG printout (snp_score.c:1545-1573)."""
    data = sim("tiny")
    cols = column_dump(["-9"], data)
    cols = cols[cols["tid"] == 0]
    exp = [l.rstrip("\n").split("\t") for l in open(GDIR / "ref_columns.tiny.-9.txt")]
    proc = cols[(cols["flags"] & 8) != 0][: len(exp)]
    assert len(proc) == len(exp)
    for c, e in zip(proc, exp):
        assert int(e[0]) == c["pos"] + 1 and int(e[1]) == c["n_plp"]
        if c["het_phred"] > 0:
            s = "%c/%c %4d" % ("ACGT*"[c["het_call"] // 5], "ACGT*"[c["het_call"] % 5], c["het_phred"])
        else:
            s = "%c   %4d" % ("ACGT*N"[c["call"]], c["phred"])
        assert e[2] == s, (e, c)
        assert (len(e) > 3 and e[3] == "*") == bool(c["flags"] & 1)


# SURVEY.md §9.5: known answers of calculate_consensus_pileup (reference lines 231-797 compiled verbatim)
KAT = [  # bases, qual, mapq, (mode A), (mode B): call, het_call, phred, het_phred, discrep
    ("A" * 30, 30, 60, (0, 1, 147, -152, 0.0), (0, 1, 146, -151, 0.0)),
    ("A" * 30, 40, 60, (0, 1, 147, -152, 0.0), (0, 1, 147, -152, 0.0)),
    ("A" * 30, 30, 20, (0, 1, 147, -152, 0.0), (0, 1, 143, -148, 0.0)),
    ("A" * 15 + "T" * 15, 30, 60, (0, 3, 0, 384, 0.0), (0, 3, 0, 142, 0.0)),
    ("A" * 29 + "C", 30, 60, (0, 1, 117, -116, 0.182483), (0, 1, 132, -131, 0.178903)),
    ("A" * 27 + "CCC", 30, 60, (0, 1, 45, -44, 0.547449), (0, 1, 92, -91, 0.536709)),
    ("A" * 5, 30, 60, (0, 1, 72, -77, 0.0), (0, 1, 72, -77, 0.0)),
    ("A" * 10, 30, 60, (0, 1, 87, -92, 0.0), (0, 1, 87, -92, 0.0)),
    ("A", 30, 60, (0, 1, 30, -65, 0.0), (0, 1, 14, -65, 0.0)),
    ("N", 30, 60, (5, 0, 0, 0, 0.0), (5, 0, 0, 0, 0.0)),
    ("AC", 30, 60, (0, 1, 0, -35, 0.706753), (0, 1, 0, -51, 0.692889)),
]


def kat_stream(bases, qual, mapq):
    """one-base reads stacked on one column, as an uncompressed BAM stream"""
    hdr = b"@SQ\tSN:k\tLN:100\n"
    out = bytearray(b"BAM\1" + struct.pack("<i", len(hdr)) + hdr + struct.pack("<i", 1) + struct.pack("<i", 2) + b"k\0" + struct.pack("<i", 100))
    code = {"A": 1, "C": 2, "G": 4, "T": 8, "N": 15}
    for i, b in enumerate(bases):
        name = b"r%d\0" % i
        rec = struct.pack("<iiBBHHHiiii", 0, 10, len(name), mapq, 4680, 1, 0, 1, -1, -1, 0) + name + struct.pack("<I", 1 << 4) + bytes([code[b] << 4]) + bytes([qual])
        out += struct.pack("<i", len(rec)) + rec
    return np.frombuffer(bytes(out), dtype=np.uint8)


@pytest.mark.parametrize("kat", KAT, ids=lambda k: f"{len(k[0])}x{k[0][0]}{k[0][-1]}q{k[1]}m{k[2]}")
def test_port_consensus_known_answers(kat):
    bases, qual, mapq, expA, expB = kat
    data = kat_stream(bases, qual, mapq)
    for args, exp in ((["-q70", "-Q0"], expA), (["-9"], expB)):
        c = column_dump(args, data)
        assert len(c) == 1
        got = (int(c[0]["call"]), int(c[0]["het_call"]), int(c[0]["phred"]), int(c[0]["het_phred"]))
        assert got == exp[:4], (args, got, exp)
        assert abs(float(c[0]["discrep"]) - exp[4]) < 5e-7
