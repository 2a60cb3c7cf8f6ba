#!/usr/bin/env python
"""Regenerates the golden fixtures from oracle/_ref (the reference's own sources compiled
verbatim: make -C oracle ref REF=<crumble source tree>).

    python tests/golden/make_golden.py
    python tests/golden/make_golden.py --oracle-runs recorded.jsonl ...

Outputs (committed):
  golden.json                      sha256 of the rewritten quality bytes, BED text and -v counters for
                                   seeded synthetic data sets (crumble_b200.simulate) at several option sets
  edge_cases.<tag>.qual.txt        rewritten quality strings of tests/golden/edge_cases.sam, one read per line
  edge_cases.<tag>.bed             BED output for the same runs
  ref_columns.tiny.-9.txt          the reference's own -DDEBUG per-column dump (call / score / preserve mark)
  oracle_runs.json                 (--oracle-runs) the vectors every default oracle run of the tests is pinned to (tests/util.py):
                                   the JSON lines that `CRUMBLE_ORACLE_RECORD=recorded.jsonl pytest tests` appends, merged, plus the
                                   sha256 of the -DDEBUG per-column lines test_gpu_columns_match_reference_debug_dump checks; made
                                   with the oracle of record (the reference when oracle/_ref is built, else the restatement), and each
                                   labelled with it ("made_by"); restatement vectors on golden.json's inputs say whether they equal
                                   the reference's vector there ("equals_reference")
"""
import hashlib
import json
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT)); sys.path.insert(0, str(ROOT / "tests"))
import numpy as np  # noqa: E402
import crumble_b200 as cb  # noqa: E402
from util import REF_BIN, run_oracle, valid_mask  # noqa: E402

SETS = {"tiny": ("tiny", 1.0, 3), "c1s": ("C1", 0.1, 11), "c2s": ("C2", 1 / 512, 5), "c4s": ("C4", 0.02, 4)}
ARGS = [["-9"], ["-8"], ["-7"], ["-5"], ["-3"], ["-1"], ["-1", "-B"], ["-9", "-Y0.1"], ["-5", "-q30"], ["-9", "-U30"],
        ["-1", "-m10", "-C0.05", "-Z0.01"], ["-9", "-p0", "-L0"], ["-9", "-X0.5", "-D200"], ["-3", "-i0.5,3", "-s2.0,1"]]
# options served by the plain per-item kernels (-S, -k/-K/-y, -N, -R); BED = tests/golden/keep.<set>.bed
OPT_SETS = ("tiny", "c1s")
OPT_ARGS = [["-9", "-S"], ["-1", "-S", "-B"], ["-9", "-k", "37"], ["-9", "-K", "11", "-k", "25"], ["-9", "-N", "-k", "25"], ["-9", "-N"],
            ["-9", "-y", "pbccs"], ["-9", "-R", "BED"], ["-1", "-R", "BED", "-p", "8"], ["-5", "-S", "-K", "37", "-N", "-R", "BED"],
            ["-1", "-q", "30", "-k", "37", "-S"]]
KEEP_BED = {"tiny": "chr1\t1000\t3000\nchr1\t2500\t2600\nchr1\t2800\t5000\n# nested + overlapping on purpose (bed.c:20-40)\nchr2\t100\t200\nchr2\t20000\t26000\nchr1\t40000\t41000\n",
            "c1s": "track name=keep\nchr20\t1000\t3000\nchr20\t2500\t2600\nchr20\t2800\t5000\nchr20\t20000\t20100\nchr20\t40000\t49000\nchr20\t90000\t90001\n"}
# aux-tag options (purge_tags, snp_score.c:989-1054): the reference's whole SAM output for tests/golden/tags.sam
TAGS = {"plain": ["-9"], "t": ["-9", "-t", "NM,BD"], "T": ["-9", "-T", "MD,XX,ZB"], "efg": ["-9", "-e", "5", "-f", "20", "-g", "40"],
        "EFGt": ["-9", "-E", "7", "-F", "25", "-G", "45", "-t", "BI,BD,RG"], "all": ["-1", "-e", "1", "-f", "30", "-g", "2", "-E", "3", "-F", "10", "-G", "50", "-T", "BI"]}
EDGE = {"l9": ["-9"], "l1B": ["-1", "-B"], "l5q30": ["-5", "-q30"], "l3U35": ["-3", "-U35", "-Y0.2"],
        "l9r": ["-9", "-r", "chrA:900-1600"], "l1r": ["-1", "-r", "chrA:1200-2100"]}


def oracle_runs(recorded):
    import hashlib as H
    import os, tempfile
    from util import STORED, oracle_bin, stored_key
    from test_gpu_parity import debug_dump_lines
    runs = {}
    for path in recorded:
        for line in open(path):
            for k, v in json.loads(line).items():
                assert runs.setdefault(k, v) == v, f"two different vectors recorded for {k!r}"
    for name, g in json.load(open(HERE / "golden.json")).items():
        data, _, _ = cb.simulate(g["preset"], g["scale"], g["seed"])
        for args, exp in g["runs"].items():
            v = runs.get(stored_key(H.sha256(data.tobytes()).hexdigest(), args.split()))
            if v is not None and v["made_by"] != "reference":
                v["equals_reference"] = v["qual_sha256"] == exp["qual_sha256"] and v["counters"] == exp["counters"] and \
                    v["bed_sha256"] == H.sha256(exp["bed"].encode()).hexdigest()
    binary, kind = oracle_bin()
    for preset, scale, seed, args in (("tiny", 1.0, 3, ["-9"]), ("C1", 0.25, 11, ["-9"]), ("C1", 0.25, 11, ["-1"])):
        data, _, _ = cb.simulate(preset, scale, seed)
        with tempfile.TemporaryDirectory() as td:
            fin, dump = os.path.join(td, "i.ubam"), os.path.join(td, "cols.bin")
            data.tofile(fin)
            if kind == "reference":
                dbg = subprocess.run([str(binary.parent / "crumble_ref_debug"), "-z"] + args + [fin, "mem:x"], stdout=subprocess.PIPE, text=True, check=True).stdout
                lines = []
                for l in dbg.splitlines():
                    if l.startswith("Depth "):
                        e = l.split("\t")
                        lines.append("\t".join([e[0].split(" ")[1]] + e[1:4] + [e[4] if len(e) > 4 and e[4] == "*" else ""]))
            else:
                subprocess.run([str(binary), "-z"] + args + [fin, "mem:x"], check=True, env=dict(os.environ, ORACLE_COLUMN_DUMP=dump))
                lines = debug_dump_lines(np.fromfile(dump, dtype=cb.api.COLUMN_DTYPE))
        runs["columns " + stored_key(H.sha256(data.tobytes()).hexdigest(), args)] = {
            "sha256": H.sha256("\n".join(lines).encode()).hexdigest(), "made_by": "reference" if kind == "reference" else "restatement"}
    with open(STORED, "w") as f:                                # one vector per line
        f.write("{\n" + ",\n".join(f"{json.dumps(k)}: {json.dumps(runs[k], sort_keys=True)}" for k in sorted(runs)) + "\n}\n")
    print(f"{len(runs)} oracle vectors written ({kind})")


def main():
    ref = ROOT / "oracle" / "_ref" / "crumble_ref"
    assert ref.exists(), "build oracle/_ref first (make -C oracle ref)"
    gold = {}
    for name, (preset, scale, seed) in SETS.items():
        data, nr, nb = cb.simulate(preset, scale, seed, threads=1)
        bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish()
        m = valid_mask(bb)
        gold[name] = {"preset": preset, "scale": scale, "seed": seed, "reads": nr, "aligned_bases": nb,
                      "input_sha256": hashlib.sha256(data.tobytes()).hexdigest(), "runs": {}}
        for a in ARGS:
            r = run_oracle(data, a, binary=REF_BIN, kind="reference")
            gold[name]["runs"][" ".join(a)] = {"qual_sha256": hashlib.sha256(r["qual"][m].tobytes()).hexdigest(),
                                               "bed": r["bed"], "counters": r["counters"]}
        if name in OPT_SETS:
            bedf = HERE / f"keep.{name}.bed"
            bedf.write_text(KEEP_BED[name])
            gold[name]["opt_runs"] = {}
            for a in OPT_ARGS:
                r = run_oracle(data, [str(bedf) if x == "BED" else x for x in a], binary=REF_BIN, kind="reference")
                gold[name]["opt_runs"][" ".join(a)] = {"qual_sha256": hashlib.sha256(r["qual"][m].tobytes()).hexdigest(),
                                                       "bed": r["bed"], "counters": r["counters"]}
        bb.close()
    json.dump(gold, open(HERE / "golden.json", "w"), indent=1, sort_keys=True)
    sam = HERE / "edge_cases.sam"
    for tag, a in EDGE.items():
        out, bed = HERE / f"_tmp.{tag}.sam", HERE / f"edge_cases.{tag}.bed"
        subprocess.run([str(ref), "-z"] + a + ["-b", str(bed), str(sam), str(out)], check=True)
        with open(HERE / f"edge_cases.{tag}.qual.txt", "w") as f:
            for line in open(out):
                if not line.startswith("@"):
                    c = line.rstrip("\n").split("\t"); f.write(c[0] + "\t" + c[10] + "\n")
        out.unlink()
    for tag, a in TAGS.items():
        subprocess.run([str(ref), "-z"] + a + [str(HERE / "tags.sam"), str(HERE / f"tags.{tag}.out.sam")], check=True)
    # the reference's own debug dump: "Depth tid pos n_plp \t call score \t[*]\t bases"
    data, _, _ = cb.simulate(*SETS["tiny"], threads=1)
    tmp = HERE / "_tmp.ubam"; data.tofile(tmp)
    dbg = subprocess.run([str(ROOT / "oracle" / "_ref" / "crumble_ref_debug"), "-z", "-9", str(tmp), "mem:x"],
                         stdout=subprocess.PIPE, text=True, check=True).stdout
    tmp.unlink()
    with open(HERE / "ref_columns.tiny.-9.txt", "w") as f:
        n = 0
        for line in dbg.splitlines():
            if line.startswith("Depth 0"):           # first contig, first 20000 columns: pos(1-based) depth call+score mark
                c = line.split("\t")
                f.write("\t".join(c[1:5]).rstrip("\t") + "\n")
                n += 1
                if n == 20000:
                    break
    print("golden fixtures written")


if __name__ == "__main__":
    if sys.argv[1:2] == ["--oracle-runs"]:
        oracle_runs(sys.argv[2:])
    else:
        main()
