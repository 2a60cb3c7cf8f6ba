"""Test helpers: run the CPU oracle on a raw BAM stream and bring its output into the
same structure-of-arrays layout the GPU path uses.

Oracle choice: oracle/_ref/crumble_ref (the reference's own sources compiled verbatim with
make -C oracle ref REF=<crumble source tree>) when it is built; otherwise "stored":
oracle/bin/crumble_oracle (this repository's plain-C restatement, which reproduces every vector
of golden.json made with the reference) pinned to tests/golden/oracle_runs.json.  Either way
the checker's output for every input and option set the parity tests use must equal the stored
vector (sha256 of the quality bytes and of the BED text, the -v counters), so a change to the
oracle cannot move the bar.  Every stored vector names the oracle that made it ("made_by":
"reference" or "restatement"); a restatement vector whose input and options golden.json also
covers says whether it equals the reference's vector there ("equals_reference").  Run with
oracle/_ref built and re-record to replace restatement vectors with the reference's own.
kind="port" runs the restatement unpinned."""
import hashlib
import json
import os
import re
import subprocess
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
REF_BIN = ROOT / "oracle" / "_ref" / "crumble_ref"
PORT_BIN = ROOT / "oracle" / "bin" / "crumble_oracle"
EMU_BIN = ROOT / "tests" / "emu" / "emu_crumble"
STORED = ROOT / "tests" / "golden" / "oracle_runs.json"


def oracle_bin(kind=None):
    """kind None = the checker of record: the verbatim reference when oracle/_ref is built, else the restatement pinned to the stored
    vectors (kind "stored"); CRUMBLE_ORACLE in the environment overrides the choice."""
    if kind is None:
        kind = os.environ.get("CRUMBLE_ORACLE") or ("reference" if REF_BIN.exists() else "stored")
    if kind == "reference":
        if REF_BIN.exists():
            return REF_BIN, "reference"
        raise FileNotFoundError(f"{REF_BIN} is missing: build it with make -C oracle ref REF=<crumble source tree>")
    if kind in ("port", "stored") and PORT_BIN.exists():
        return PORT_BIN, kind
    raise FileNotFoundError("no oracle binary: run __graft_entry__.build()")


def stored_key(data_sha256, args):
    return data_sha256 + " " + " ".join(args)


def pin_to_stored(res, data_sha256, args, mask):
    """The oracle's result for this input (sha256 of the uncompressed BAM stream) and these options must equal the stored vector.
    With CRUMBLE_ORACLE_RECORD=<file> the vector is appended to that file (JSON lines) instead, to extend oracle_runs.json."""
    got = {"qual_sha256": hashlib.sha256(res["qual"][mask].tobytes()).hexdigest(),
           "bed_sha256": hashlib.sha256(res["bed"].encode()).hexdigest(), "counters": res["counters"]}
    key = stored_key(data_sha256, args)
    rec = os.environ.get("CRUMBLE_ORACLE_RECORD")
    if rec:
        with open(rec, "a") as f:
            f.write(json.dumps({key: dict(got, made_by="reference" if res["kind"] == "reference" else "restatement")}, sort_keys=True) + "\n")
        return
    exp = json.load(open(STORED)).get(key)
    assert exp is not None, f"no stored oracle vector for {key!r} in {STORED.name}"
    assert got == {k: exp[k] for k in got}, \
        f"the oracle ({res['kind']}) does not reproduce the stored vector for {key!r} (made by the {exp['made_by']})"
    res["kind"] = f"{res['kind']}, pinned to a vector made by the {exp['made_by']}"


def parse_counters(stderr_text):
    import crumble_b200 as cb
    pats = {
        "diff": r"A/B Diff\s+= (\d+)", "indel_pair": r"A/B Indel\s+= (\d+) / (\d+)",
        "hetA": r"A:  Het\s+= (\d+) / (\d+)", "homA": r"A:  Hom\s+= (\d+) / (\d+)", "discA": r"A:  Discrep\s+= (\d+)",
        "hetB": r"B:  Het\s+= (\d+) / (\d+)", "homB": r"B:  Hom\s+= (\d+) / (\d+)", "discB": r"B:  Discrep\s+= (\d+)",
        "columns": r"Columns\s+= (\d+)", "low_mqual_perc": r"Low_mqual_perc\s+= (\d+)", "clip_perc": r"Clip_perc\s+= (\d+)",
        "ins_len_perc": r"Ins_len_perc\s+= (\d+)", "indel_ov_perc": r"indel_ov_perc\s+= (\d+)", "over_depth": r"count_over_depth = (\d+)",
    }
    g = {k: re.search(p, stderr_text) for k, p in pats.items()}
    if not all(g.values()):
        return None
    return {
        "diff": int(g["diff"][1]), "indel_qual": int(g["indel_pair"][1]), "indel": int(g["indel_pair"][2]),
        "het_qual_A": int(g["hetA"][1]), "het_A": int(g["hetA"][2]), "hom_qual_A": int(g["homA"][1]), "hom_A": int(g["homA"][2]),
        "discrep_A": int(g["discA"][1]), "het_qual_B": int(g["hetB"][1]), "het_B": int(g["hetB"][2]),
        "hom_qual_B": int(g["homB"][1]), "hom_B": int(g["homB"][2]), "discrep_B": int(g["discB"][1]),
        "columns": int(g["columns"][1]), "low_mqual_perc": int(g["low_mqual_perc"][1]), "clip_perc": int(g["clip_perc"][1]),
        "ins_len_perc": int(g["ins_len_perc"][1]), "indel_ov_perc": int(g["indel_ov_perc"][1]), "over_depth": int(g["over_depth"][1]),
    }


def header_names(data: np.ndarray):
    b = data.tobytes()[: 1 << 20]
    lt = int.from_bytes(b[4:8], "little")
    p = 8 + lt
    n = int.from_bytes(b[p:p + 4], "little"); p += 4
    names = []
    for _ in range(n):
        ln = int.from_bytes(b[p:p + 4], "little"); p += 4
        names.append(b[p:p + ln - 1].decode()); p += ln + 4
    return names


def run_oracle(data: np.ndarray, args, kind=None, binary=None, timing=False, env_extra=None):
    """Run the oracle CLI on an uncompressed BAM stream; returns quals in batch layout, BED text, counters."""
    import crumble_b200 as cb
    pinned = binary is None and kind in (None, "reference", "stored")
    if binary is None:
        binary, kind = oracle_bin(kind)
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        fin, fout, fbed = os.path.join(td, "in.ubam"), os.path.join(td, "out.ubam"), os.path.join(td, "out.bed")
        data.tofile(fin)
        env = dict(os.environ)
        env["CRUMBLE_REF_TIMING"] = "1"
        env.update(env_extra or {})
        cmd = [str(binary), "-z", "-v"] + list(args) + ["-b", fbed, "-O", "bam,raw", fin, fout]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
        if r.returncode != 0:
            raise RuntimeError(f"oracle failed ({r.returncode}): {r.stderr[-2000:]}")
        out = np.fromfile(fout, dtype=np.uint8)
        bed = open(fbed).read()
    bb = cb.BatchBuilder(pinned=False)
    bb.add_bam_stream(out)
    bb.finish()
    m = re.search(r"transcode_seconds=([0-9.]+)", r.stderr)
    res = {"qual": bb.qual().copy(), "pos": bb.positions(), "len": bb.lengths(), "off": bb.offsets(), "bed": bed, "counters": parse_counters(r.stderr), "names": header_names(data),
           "kind": kind, "seconds": float(m[1]) if m else None, "stderr": r.stderr}
    if pinned:
        pin_to_stored(res, hashlib.sha256(data.tobytes()).hexdigest(), args, valid_mask(bb))
    bb.close()
    return res


def valid_mask(bb):
    """Boolean mask over the padded quality buffer selecting real quality bytes."""
    off, ln = bb.offsets(), bb.lengths()
    total = int(bb.batch.qual_bytes)
    m = np.zeros(total + 1, dtype=np.int32)
    np.add.at(m, off, 1)
    np.add.at(m, off + ln, -1)
    return np.cumsum(m[:-1]) > 0


def add_ambiguity_codes(data: np.ndarray, rate: float, seed: int = 1):
    """a copy of an uncompressed BAM stream with a fraction of the bases replaced by N (mostly), other ambiguity codes and '='"""
    import struct
    d = data.copy(); rng = np.random.default_rng(seed)
    b = d.tobytes(); p = 8 + struct.unpack_from('<i', b, 4)[0]
    nref = struct.unpack_from('<i', b, p)[0]; p += 4
    for _ in range(nref):
        p += 4 + struct.unpack_from('<i', b, p)[0] + 4
    n = 0
    while p + 4 <= len(b):
        bs = struct.unpack_from('<i', b, p)[0]; r = p + 4
        lname = b[r + 8]; ncig = struct.unpack_from('<H', b, r + 12)[0]; lseq = struct.unpack_from('<i', b, r + 16)[0]
        so = r + 32 + lname + 4 * ncig
        for x in rng.integers(0, max(lseq, 1), rng.binomial(lseq, rate) if lseq else 0):
            code = [15, 15, 15, 3, 0, 14][rng.integers(0, 6)]
            i = so + (int(x) >> 1)
            d[i] = (d[i] & 0xf0) | code if x & 1 else (d[i] & 0x0f) | (code << 4)
            n += 1
        p += 4 + bs
    return d, n
