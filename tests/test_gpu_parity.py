"""GPU parity tests proper: the CUDA path, called through the C ABI, against the CPU oracle
on the same seeded inputs.  Bar: quality strings, BED events and -v counters bit-exact."""
import numpy as np
import pytest

import crumble_b200 as cb
from util import run_oracle, valid_mask

pytestmark = pytest.mark.gpu

LEVELS = [["-9"], ["-8"], ["-7"], ["-5"], ["-3"], ["-1"], ["-1", "-B"], ["-9", "-Y0.1"], ["-5", "-q30"],
          ["-9", "-U30"], ["-1", "-m10", "-C0.05", "-Z0.01"]]


def params_from_args(args):
    """Python mirror of the reference getopt loop for the options the tests use."""
    p = cb.default_params()
    lib = cb.load_lib()
    import ctypes as C
    for a in args:
        k, v = a[1], a[2:]
        if k in "135789":
            lib.cg_params_level(C.byref(p), int(k))
        elif k == "B": p.binary_qual = 1
        elif k == "Y": p.indel_fract = float(v)
        elif k == "q": p.min_qual_A = int(v)
        elif k == "Q": p.min_qual_B = int(v)
        elif k == "U": p.qcap = int(v)
        elif k == "m": p.min_mqual = int(v)
        elif k == "C": p.clip_perc = float(v)
        elif k == "Z": p.ins_len_perc = float(v)
        elif k == "P": p.over_depth = float(v)
        elif k == "p": p.pblock = int(v)
        elif k == "L": p.reduce_qual = int(v)
        elif k == "D": p.min_indel_B = int(v)
        elif k == "X": p.min_discrep_B = float(v)
        else: raise ValueError(a)
    return p


_cache = {}


def dataset(name):
    if name not in _cache:
        preset, scale, seed = {"tiny": ("tiny", 1.0, 3), "c1s": ("C1", 0.25, 11), "c2s": ("C2", 1 / 128, 5), "c4s": ("C4", 0.05, 4),
                               "c4m": ("C4", 0.15, 6)}[name]       # c4m: 30 amplicons, enough for STR triggers and indel spectra to fire at 1000x
        data, nr, nb = cb.simulate(preset, scale, seed)
        bb = cb.BatchBuilder()
        bb.add_bam_stream(data)
        batch = bb.finish()
        _cache[name] = (data, bb, batch, valid_mask(bb))
    return _cache[name]


def check(name, args, chunk_bytes=None):
    data, bb, batch, mask = dataset(name)
    g = cb.Crumble(params_from_args(args), device=0)
    if chunk_bytes:
        g.set_chunk_bytes(chunk_bytes)
    out = g.process(batch)
    ref = run_oracle(data, args)
    nbad = int((out["qual"][mask] != ref["qual"][mask]).sum())
    assert nbad == 0, f"{nbad} quality bytes differ from the oracle ({ref['kind']})"
    assert cb.bed_text(out["events"], ref["names"]) == ref["bed"]
    assert out["counters"] == ref["counters"]
    g.close()


@pytest.mark.parametrize("args", LEVELS, ids=lambda a: "".join(a))
def test_tiny_all_levels(args):
    check("tiny", args)


@pytest.mark.parametrize("name", ["c1s", "c2s", "c4s", "c4m"])
@pytest.mark.parametrize("args", [["-9"], ["-1", "-B"], ["-5"]], ids=lambda a: "".join(a))
def test_configs(name, args):
    check(name, args)


@pytest.mark.parametrize("name,args", [("c4m", ["-9", "-D300"]), ("c4m", ["-1", "-D300", "-X0.2"]), ("c4s", ["-1", "-D300", "-Q300"])],
                         ids=lambda v: "".join(v) if isinstance(v, list) else v)
def test_str_triggers_at_depth(name, args):
    """1000x amplicon columns never score below the default indel threshold, so the C4 workload alone runs no STR search at all: -D300 makes
    every indel column a trigger (a thousand reads each), -Q300 at -1 preserves every column so that EVERY read of every column triggers
    (str_snp && preserve, snp_score.c:1718): the item list, the list-free search and the window chain under the heaviest load the options
    allow, against the oracle"""
    check(name, args)
    check(name, args, chunk_bytes=1 << 18)


@pytest.mark.parametrize("name,chunk", [("tiny", 1 << 16), ("c1s", 1 << 20), ("c2s", 1 << 18), ("c4s", 1 << 17), ("c1s", 3 << 18)])
@pytest.mark.parametrize("args", [["-9"], ["-1"], ["-1", "-B"], ["-3", "-P1.5"], ["-5", "-q30"]], ids=lambda a: "".join(a))
def test_streamed_slices(name, chunk, args):
    """cg_process cut into many upload chunks / slices (keep-window chain, depth average and BED order carried
    across slices on the device) gives the oracle's bytes, events and counters."""
    check(name, args, chunk_bytes=chunk)


def test_resident_equals_streamed():
    """upload + run + download (one slice) and the streamed cg_process agree byte for byte."""
    data, bb, batch, mask = dataset("c1s")
    g = cb.Crumble(params_from_args(["-1"]), device=0)
    g.set_chunk_bytes(1 << 19)
    a = g.process(batch)
    g.upload(batch); g.run()
    b = g.download(batch)
    assert np.array_equal(a["qual"][mask], b["qual"][mask])
    assert np.array_equal(a["events"], b["events"]) and a["counters"] == b["counters"]
    g.close()


def test_smoke_entry():
    import __graft_entry__ as g
    g.smoke()


# ---- golden vectors (generated from the verbatim reference; no oracle run needed) --------------
import hashlib
import json
import os
import subprocess
import tempfile

from util import ROOT, PORT_BIN

GOLD = json.load(open(ROOT / "tests" / "golden" / "golden.json"))
GDIR = ROOT / "tests" / "golden"


@pytest.mark.parametrize("name", sorted(GOLD))
def test_gpu_matches_golden(name):
    g0 = GOLD[name]
    data, nr, nb = cb.simulate(g0["preset"], g0["scale"], g0["seed"], threads=2)
    assert hashlib.sha256(data.tobytes()).hexdigest() == g0["input_sha256"]
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish(); m = valid_mask(bb)
    names = ["chr20"] if g0["preset"] != "tiny" else ["chr1", "chr2"]
    for args, exp in g0["runs"].items():
        p = cb.default_params()
        import ctypes as C
        for a in args.split():
            k, v = a[1], a[2:]
            if k in "135789": cb.load_lib().cg_params_level(C.byref(p), int(k))
            elif k == "B": p.binary_qual = 1
            elif k == "Y": p.indel_fract = float(v)
            elif k == "q": p.min_qual_A = int(v)
            elif k == "U": p.qcap = int(v)
            elif k == "m": p.min_mqual = int(v)
            elif k == "C": p.clip_perc = float(v)
            elif k == "Z": p.ins_len_perc = float(v)
            elif k == "p": p.pblock = int(v)
            elif k == "L": p.reduce_qual = int(v)
            elif k == "X": p.min_discrep_B = float(v)
            elif k == "D": p.min_indel_B = int(v)
            elif k == "i": p.iSTR_mul = float(v.split(",")[0]); p.iSTR_add = int(v.split(",")[1])
            elif k == "s": p.sSTR_mul = float(v.split(",")[0]); p.sSTR_add = int(v.split(",")[1])
            else: raise ValueError(a)
        g = cb.Crumble(p, device=0)
        out = g.process(batch)
        assert hashlib.sha256(out["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"], args
        assert cb.bed_text(out["events"], names) == exp["bed"], args
        assert out["counters"] == exp["counters"], args
        g.close()


EDGE = {"l9": ["-9"], "l1B": ["-1", "-B"], "l5q30": ["-5", "-q30"], "l3U35": ["-3", "-U35", "-Y0.2"],
        "l9r": ["-9", "-r", "chrA:900-1600"], "l1r": ["-1", "-r", "chrA:1200-2100"]}

OPT = [(n, a) for n in sorted(GOLD) for a in sorted(GOLD[n].get("opt_runs", {}))]


@pytest.mark.parametrize("name,args", OPT, ids=lambda v: v.replace(" ", "") if isinstance(v, str) else None)
def test_gpu_cli_options(name, args):
    """-S, -k/-K/-y pbccs, -N, -R keep.bed through the crumble_gpu command line (option parsing, bed loading, host driver,
    device path with the plain per-item kernels) against golden vectors made with the verbatim reference."""
    g0 = GOLD[name]
    data, nr, nb = cb.simulate(g0["preset"], g0["scale"], g0["seed"], threads=2)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish(); m = valid_mask(bb)
    exp = g0["opt_runs"][args]
    argv = [str(GDIR / f"keep.{name}.bed") if x == "BED" else x for x in args.split()]
    r = run_oracle(data, argv, binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli")
    assert hashlib.sha256(r["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"]
    assert r["bed"] == exp["bed"]
    assert r["counters"] == exp["counters"]


@pytest.mark.parametrize("tag", sorted(EDGE))
def test_gpu_cli_edge_cases(tag):
    """the crumble_gpu command line (host driver + device path) on the odd-CIGAR SAM, against the reference's output"""
    cli = ROOT / "crumble_b200" / "lib" / "crumble_gpu"
    with tempfile.TemporaryDirectory() as td:
        out, bed = os.path.join(td, "o.sam"), os.path.join(td, "o.bed")
        r = subprocess.run([str(cli), "-z"] + EDGE[tag] + ["-b", bed, str(GDIR / "edge_cases.sam"), out], stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        quals = [(l.rstrip("\n").split("\t")[0], l.rstrip("\n").split("\t")[10]) for l in open(out) if not l.startswith("@")]
        exp = [tuple(l.rstrip("\n").split("\t")) for l in open(GDIR / f"edge_cases.{tag}.qual.txt")]
        assert quals == exp
        assert open(bed).read() == open(GDIR / f"edge_cases.{tag}.bed").read()
        # aux tags and everything else pass through untouched; @PG is added without -z
        r = subprocess.run([str(cli), "-9", str(GDIR / "edge_cases.sam"), out], stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0
        txt = open(out).read()
        assert "@PG\tID:crumble\tPN:crumble\tVN:0.9.1" in txt and "XX:Z:keepme" in txt


def test_gpu_columns_bit_exact():
    """per-column consensus (call, het_call, phred, het_phred, discrep) and column decisions against the CPU oracle:
    the tolerance north_star allows is not needed — every field, including the float discrepancy, is identical."""
    data, bb, batch, mask = dataset("c1s")
    for args in (["-9"], ["-1"]):
        g = cb.Crumble(params_from_args(args), device=0)
        out = g.process(batch, want_columns=True)
        cols = out["columns"]
        with tempfile.TemporaryDirectory() as td:
            fin, dump = os.path.join(td, "i.ubam"), os.path.join(td, "cols.bin")
            data.tofile(fin)
            subprocess.run([str(PORT_BIN), "-z"] + args + [fin, "mem:x"], check=True, env=dict(os.environ, ORACLE_COLUMN_DUMP=dump))
            exp = np.fromfile(dump, dtype=cb.api.COLUMN_DTYPE)
        assert len(cols) == len(exp)
        for f in ("tid", "pos", "n_plp", "call", "het_call", "phred", "het_phred"):
            assert np.array_equal(cols[f], exp[f]), f
        assert np.array_equal(cols["discrep"].view(np.uint32), exp["discrep"].view(np.uint32)), "discrep differs bitwise"
        for bit, nm in ((1, "preserve"), (2, "keep_qual"), (4, "window active"), (8, "processed")):
            assert np.array_equal(cols["flags"] & bit, exp["flags"] & bit), nm
        assert np.array_equal((cols["flags"] >> 8) & 31, (exp["flags"] >> 8) & 31), "BED tags"
        g.close()


def debug_dump_lines(cols):
    """processed columns as the reference's -DDEBUG printout shows them (snp_score.c:1545-1573): tid, position, depth, call or het call
    with its score, preserve mark"""
    proc = cols[(cols["flags"] & 8) != 0]
    out = []
    for c in proc:
        s = ("%c/%c %4d" % ("ACGT*"[c["het_call"] // 5], "ACGT*"[c["het_call"] % 5], c["het_phred"])) if c["het_phred"] > 0 else ("%c   %4d" % ("ACGT*N"[c["call"]], c["phred"]))
        out.append("%d\t%d\t%d\t%s\t%s" % (c["tid"], c["pos"] + 1, c["n_plp"], s, "*" if c["flags"] & 1 else ""))
    return out


@pytest.mark.parametrize("name,args", [("tiny", ["-9"]), ("c1s", ["-9"]), ("c1s", ["-1"])], ids=lambda v: "".join(v) if isinstance(v, list) else v)
def test_gpu_columns_match_reference_debug_dump(name, args):
    """the same per-column dump against the REFERENCE's own -DDEBUG printout (snp_score.c:1545-1573; oracle/_ref/crumble_ref_debug,
    compiled from the reference's sources): position, depth, call or het call, score, and the preserve mark, for every processed column.
    Without oracle/_ref: tiny -9 is checked against the reference's printout stored in tests/golden/ref_columns.tiny.-9.txt (the first
    20000 processed columns of chr1), and every case's whole printout against its stored sha256 in tests/golden/oracle_runs.json (key
    "columns <input> <options>"), which names the oracle that made it; the c1s hashes were made by the restatement, so for c1s this is a
    check against the restatement pinned in the repository, not against the reference."""
    from util import REF_BIN, STORED, stored_key
    dbg_bin = REF_BIN.parent / "crumble_ref_debug"
    data, bb, batch, mask = dataset(name)
    g = cb.Crumble(params_from_args(args), device=0)
    cols = g.process(batch, want_columns=True)["columns"]
    g.close()
    got = debug_dump_lines(cols)
    assert len(got) > 1000
    if not dbg_bin.exists():
        ref_file = GDIR / f"ref_columns.{name}.{''.join(args)}.txt"
        if ref_file.exists():
            exp = [l.rstrip("\n").split("\t") for l in open(ref_file)]
            chr1 = [c.split("\t")[1:] for c in got if c.startswith("0\t")][: len(exp)]
            assert len(chr1) == len(exp)
            for e, c in zip(exp, chr1):
                assert e[:3] + [e[3] if len(e) > 3 else ""] == c, (e, c)
        exp = json.load(open(STORED))["columns " + stored_key(hashlib.sha256(data.tobytes()).hexdigest(), args)]
        assert hashlib.sha256("\n".join(got).encode()).hexdigest() == exp["sha256"], f"differs from the printout stored by the {exp['made_by']}"
        return
    with tempfile.TemporaryDirectory() as td:
        fin = os.path.join(td, "i.ubam"); data.tofile(fin)
        txt = subprocess.run([str(dbg_bin), "-z"] + args + [fin, "mem:x"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, check=True).stdout
    exp = [l.split("\t") for l in txt.splitlines() if l.startswith("Depth ")]
    assert len(got) == len(exp)
    for e, c in zip(exp, got):
        assert [e[0].split(" ")[1]] + e[1:4] + [e[4] if len(e) > 4 and e[4] == "*" else ""] == c.split("\t"), (e, c)


def test_gpu_contig_sharding_invariance():
    """size-independent property behind the multi-GPU split: contigs are independent, so processing a
    two-contig batch equals processing each contig on its own (this is what one-shard-per-GPU relies on)."""
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(cb.default_params(1), device=0)
    whole = g.process(batch)
    n = int(batch.n_reads)
    tid = np.ctypeslib.as_array(batch.tid, shape=(n,)); pos = np.ctypeslib.as_array(batch.pos, shape=(n,))
    flag = np.ctypeslib.as_array(batch.flag, shape=(n,)); mapq = np.ctypeslib.as_array(batch.mapq, shape=(n,))
    ln = bb.lengths(); off = bb.offsets(); nc = np.ctypeslib.as_array(batch.n_cigar, shape=(n,)); co = np.ctypeslib.as_array(batch.cigar_off, shape=(n,))
    cig = np.ctypeslib.as_array(batch.cigar, shape=(int(batch.n_cigar_total),)); seq = np.ctypeslib.as_array(batch.seq, shape=(int(batch.seq_bytes),))
    qual = bb.qual()
    ev_parts, cnt = [], None
    for t in (0, 1):
        sb = cb.BatchBuilder()
        idx = np.nonzero(tid == t)[0]
        for i in idx:
            sb.add(int(tid[i]), int(pos[i]), int(flag[i]), int(mapq[i]), cig[co[i]:co[i] + nc[i]], seq[off[i] // 2: off[i] // 2 + (ln[i] + 1) // 2], qual[off[i]: off[i] + ln[i]])
        b2 = sb.finish()
        o2 = g.process(b2)
        so = sb.offsets()
        for k, i in enumerate(idx):
            assert np.array_equal(o2["qual"][so[k]: so[k] + ln[i]], whole["qual"][off[i]: off[i] + ln[i]])
        ev_parts.append(o2["events"])
        cnt = o2["counters"] if cnt is None else {k: cnt[k] + v for k, v in o2["counters"].items()}
    assert np.array_equal(np.concatenate(ev_parts), whole["events"])
    assert cnt == whole["counters"]
    g.close()


def test_gpu_empty_and_degenerate_batches():
    g = cb.Crumble(cb.default_params(9), device=0)
    e = cb.BatchBuilder(); out = g.process(e.finish())
    assert len(out["events"]) == 0 and out["counters"]["columns"] == 0
    # only unplaced / unmapped records: everything passes through, P-block still applied (snp_score.c:2004-2005)
    u = cb.BatchBuilder()
    q = np.array([30, 31, 32, 10, 11, 40, 40, 2], np.uint8)
    u.add(-1, -1, 4, 0, np.zeros(0, np.uint32), np.zeros(4, np.uint8), q)
    u.add(0, 10, 4, 0, np.zeros(0, np.uint32), np.zeros(4, np.uint8), q)
    out = g.process(u.finish())
    assert out["counters"]["columns"] == 0
    assert list(out["qual"][:8]) == [31, 31, 31, 10, 10, 40, 40, 2] and list(out["qual"][8:16]) == [31, 31, 31, 10, 10, 40, 40, 2]
    g.close()


CHAIN = [("tiny", 97), ("c1s", 1500), ("c1s", 20000), ("c2s", 4000), ("c4s", 333)]


@pytest.mark.parametrize("name,batch", CHAIN, ids=lambda v: str(v))
def test_gpu_chained_calls(name, batch):
    """cg_process_window through the crumble_gpu command line: the stream cut every `batch` records (region shards with a
    read halo, replayed columns, keep-window and depth-average state carried on the device) must reproduce the golden
    vectors of the uncut run bit for bit: qualities, BED lines, counters."""
    g0 = GOLD[name]
    data, nr, nb = cb.simulate(g0["preset"], g0["scale"], g0["seed"], threads=2)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish(); m = valid_mask(bb)
    for args in ["-9", "-1", "-3", "-5 -q30", "-1 -m10 -C0.05 -Z0.01", "-3 -i0.5,3 -s2.0,1"]:
        exp = g0["runs"][args]
        r = run_oracle(data, args.split(), binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli",
                       env_extra={"CRUMBLE_BATCH_READS": str(batch)})
        assert hashlib.sha256(r["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"], args
        assert r["bed"] == exp["bed"], args
        assert r["counters"] == exp["counters"], args


@pytest.mark.parametrize("batch", [1, 5, 40])
def test_gpu_chained_calls_edge_cases(batch):
    cli = ROOT / "crumble_b200" / "lib" / "crumble_gpu"
    env = dict(os.environ, CRUMBLE_BATCH_READS=str(batch))
    for tag in ("l9", "l1B", "l5q30", "l3U35"):
        with tempfile.TemporaryDirectory() as td:
            out, bed = os.path.join(td, "o.sam"), os.path.join(td, "o.bed")
            r = subprocess.run([str(cli), "-z"] + EDGE[tag] + ["-b", bed, str(GDIR / "edge_cases.sam"), out], stderr=subprocess.PIPE, text=True, env=env)
            assert r.returncode == 0, r.stderr
            quals = [(l.rstrip("\n").split("\t")[0], l.rstrip("\n").split("\t")[10]) for l in open(out) if not l.startswith("@")]
            exp = [tuple(l.rstrip("\n").split("\t")) for l in open(GDIR / f"edge_cases.{tag}.qual.txt")]
            assert quals == exp, tag
            assert open(bed).read() == open(GDIR / f"edge_cases.{tag}.bed").read(), tag


def test_gpu_chained_calls_event_buffer_regrow():
    g0 = GOLD["c1s"]
    data, nr, nb = cb.simulate(g0["preset"], g0["scale"], g0["seed"], threads=2)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish(); m = valid_mask(bb)
    exp = g0["runs"]["-1"]
    r = run_oracle(data, ["-1"], binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli",
                   env_extra={"CRUMBLE_BATCH_READS": "6000", "CRUMBLE_EVENTS_CAP": "1"})
    assert hashlib.sha256(r["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"]
    assert r["bed"] == exp["bed"] and r["counters"] == exp["counters"]


def test_gpu_small_event_buffer_is_refetched_not_rerun():
    """More BED events than the caller's buffer holds: the list is fetched again from the device (cg_download), the call is not repeated."""
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_args(["-1"]), device=0)
    ref = g.process(batch)
    assert len(ref["events"]) > 1
    g2 = cb.Crumble(params_from_args(["-1"]), device=0)
    out = g2.process(batch, events_cap=1)
    assert np.array_equal(out["events"], ref["events"]) and out["counters"] == ref["counters"]
    assert np.array_equal(out["qual"][mask], ref["qual"][mask])
    assert g2._events_hint == len(ref["events"])


def test_gpu_chained_calls_options():
    g0 = GOLD["tiny"]
    data, nr, nb = cb.simulate(g0["preset"], g0["scale"], g0["seed"], threads=2)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish(); m = valid_mask(bb)
    for args, exp in g0["opt_runs"].items():
        argv = [str(GDIR / "keep.tiny.bed") if x == "BED" else x for x in args.split()]
        r = run_oracle(data, argv, binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli", env_extra={"CRUMBLE_BATCH_READS": "211"})
        assert hashlib.sha256(r["qual"][m].tobytes()).hexdigest() == exp["qual_sha256"], args
        assert r["bed"] == exp["bed"], args
        assert r["counters"] == exp["counters"], args


@pytest.mark.parametrize("name,n_shards", [("c1s", 4), ("tiny", 5), ("c2s", 8), ("c4s", 3)])
@pytest.mark.parametrize("args", [["-9"], ["-1"], ["-3", "-P1.5"]], ids=lambda a: "".join(a))
def test_gpu_region_shards_on_independent_contexts(name, n_shards, args):
    """Region shards of one batch on independent contexts, every shard started from the reset state (as it would on its own
    GPU), states checked afterwards in position order (cg_carry_export / cg_carry_is_neutral / cg_carry_import): identical
    to one call on the whole batch.  At -1/-3 the depth average is in play, so the check must fall back to the ordered chain."""
    data, bb, batch, mask = dataset(name)
    p = params_from_args(args)
    whole = cb.Crumble(p, device=0)
    ref = whole.process(batch)
    orc = run_oracle(data, args)                                    # the shards are compared with the ORACLE, not only with the single call
    ctxs = [cb.Crumble(p, device=0) for _ in range(n_shards)]
    out = cb.run_region_shards(ctxs, batch, n_shards)
    assert int((out["qual"][mask] != orc["qual"][mask]).sum()) == 0
    assert cb.bed_text(out["events"], orc["names"]) == orc["bed"] and out["counters"] == orc["counters"]
    assert np.array_equal(out["qual"][mask], ref["qual"][mask])
    assert np.array_equal(out["events"], ref["events"])
    assert out["counters"] == ref["counters"]
    # and the same shards as an ordered chain on ONE context
    seq = cb.run_region_shards([whole], batch, n_shards)
    assert np.array_equal(seq["qual"][mask], ref["qual"][mask]) and seq["counters"] == ref["counters"]
    for g in ctxs + [whole]:
        g.close()


def test_gpu_packed_and_unpacked_batches_agree():
    """cg_batch.packed = 1 (the batcher's layout): the two offset arrays are rebuilt on the device by scans instead of being
    uploaded; a caller's own layout (packed = 0) takes them from the host.  Same results, 12 bytes per record less to copy."""
    data, bb, batch, mask = dataset("c1s")
    assert batch.packed == 1
    g = cb.Crumble(params_from_args(["-9"]), device=0)
    a = g.process(batch); up_packed = g.h2d_bytes()
    loose = cb.api.Batch.from_buffer_copy(batch); loose.packed = 0
    b = g.process(loose); up_loose = g.h2d_bytes()
    assert np.array_equal(a["qual"][mask], b["qual"][mask]) and a["counters"] == b["counters"] and np.array_equal(a["events"], b["events"])
    assert up_loose - up_packed == 12 * int(batch.n_reads)
    g.upload(loose); g.run(); c = g.download(loose)
    assert np.array_equal(a["qual"][mask], c["qual"][mask])
    g.close()


@pytest.mark.parametrize("depth", [1.2, 3.0])
def test_gpu_chained_calls_sparse_coverage(depth):
    """1-3x coverage with placed-unmapped reads, cut after every record (and every 7): coverage gaps, window calls without a single
    pileup column, and at -1 / -P1.5 a depth average that must survive all of them on the device"""
    data, nr, nb = cb.simulate("tiny", 3.0, seed=17, depth=depth, features_per_mb=200.0)
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data); bb.finish(); m = valid_mask(bb)
    for args in (["-9"], ["-1"], ["-3", "-P1.5"]):
        ref = run_oracle(data, args)
        for batch in ("1", "7"):
            r = run_oracle(data, args, binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli", env_extra={"CRUMBLE_BATCH_READS": batch})
            assert (r["qual"][m] == ref["qual"][m]).all() and r["bed"] == ref["bed"] and r["counters"] == ref["counters"], (args, batch)


@pytest.mark.parametrize("name,args,chunk", [("c2s", ["-9"], 1 << 18), ("c2s", ["-1", "-B"], None), ("c1s", ["-9"], 1 << 19), ("tiny", ["-3", "-P1.5"], 1 << 16), ("c4s", ["-9"], None)],
                         ids=lambda v: "".join(v) if isinstance(v, list) else str(v))
def test_gpu_compact_planes(name, args, chunk):
    """cg_batch with the compact planes (2-bit bases + exceptions, dictionary-coded qualities): the device expands them into its
    working arrays; results equal the oracle's, resident and streamed, and the upload shrinks"""
    data, bb0, batch0, mask = dataset(name)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish(pack=True)
    g = cb.Crumble(params_from_args(args), device=0)
    if chunk:
        g.set_chunk_bytes(chunk)
    out = g.process(batch); up_packed = g.h2d_bytes()
    ref = run_oracle(data, args)
    assert int((out["qual"][mask] != ref["qual"][mask]).sum()) == 0
    assert cb.bed_text(out["events"], ref["names"]) == ref["bed"] and out["counters"] == ref["counters"]
    g.process(batch0); up_plain = g.h2d_bytes()
    saved = int(batch.qual_bytes) // 4 + (int(batch.qual_bytes) * (8 - batch.qual_bits) // 8 if batch.qual_bits else 0) - 8 * int(batch.n_seq_exc)
    assert batch.meta_planes == 1                                   # and the per-record arrays travel as compact planes too
    n = int(batch.n_reads)
    saved += n * (4 + 4 + 2 + 1 + 4 + 2) + 4 * int(batch.n_cigar_total) \
        - (n * (1 + 1 + 1 + 2 + 1) + 8 * (int(batch.n_tid_runs) + int(batch.n_pos_abs)) + 1024 + 4 * int(batch.n_cigar_x))
    assert up_plain - up_packed == saved
    g.upload(batch); g.run(); res = g.download(batch)
    assert np.array_equal(res["qual"][mask], out["qual"][mask]) and res["counters"] == out["counters"]
    # region shards carry their share of the planes
    ctxs = [cb.Crumble(params_from_args(args), device=0) for _ in range(3)]
    sh = cb.run_region_shards(ctxs, batch, 3)
    assert np.array_equal(sh["qual"][mask], out["qual"][mask]) and sh["counters"] == out["counters"]
    for c in ctxs + [g]:
        c.close()
    bb.close()


@pytest.mark.parametrize("name,rate", [("tiny", 0.01), ("c4s", 0.002), ("c1s", 0.05)])
def test_gpu_ambiguity_codes(name, rate):
    """N and other non-ACGT codes: an N adds to 14 of the 15 genotype sums (snp_score.c:677-682), which the column kernel does in
    rank space after handing every base a rank; the STR search maps them to 'A'; the compact planes list them as exceptions"""
    from util import add_ambiguity_codes
    data0 = dataset(name)[0]
    data, n = add_ambiguity_codes(data0, rate, seed=7)
    assert n > 1000
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish(pack=True); mask = valid_mask(bb)
    assert int(batch.n_seq_exc) > 0
    for args in (["-9"], ["-1", "-B"], ["-3"]):
        g = cb.Crumble(params_from_args(args), device=0)
        out = g.process(batch, want_columns=(args == ["-9"]))
        ref = run_oracle(data, args)
        assert int((out["qual"][mask] != ref["qual"][mask]).sum()) == 0, args
        assert cb.bed_text(out["events"], ref["names"]) == ref["bed"] and out["counters"] == ref["counters"], args
        g.close()
    bb.close()


@pytest.mark.parametrize("name,n_dev", [("c1s", 4), ("tiny", 5), ("c2s", 8), ("c4s", 3), ("tiny", 1)])
@pytest.mark.parametrize("args", [["-9"], ["-1"], ["-1", "-B"], ["-3", "-P1.5"], ["-5", "-q30"]], ids=lambda a: "".join(a))
def test_gpu_multi_device_scheduler(name, n_dev, args):
    """cgm_process (crumble_b200/csrc/cg_multi.c): one batch cut into as many region shards as "devices" (here: contexts on one GPU),
    state-free part on all shards at once, the true 128-byte state passed from shard to shard (cg_shard_begin / _carry / _end), every
    shard downloading its own byte range of the shared output.  No speculation, so -1 / -3 (depth average in play) run concurrently
    too.  Compared with the ORACLE, with plain and with compact-plane batches."""
    data, bb0, batch0, mask = dataset(name)
    ref = run_oracle(data, args)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); packed = bb.finish(pack=True)
    m = cb.MultiCrumble(params_from_args(args), devices=[0] * n_dev)
    assert m.n_devices() == n_dev
    for batch in (batch0, packed):
        out = m.process(batch)
        nbad = int((out["qual"][mask] != ref["qual"][mask]).sum())
        assert nbad == 0, f"{nbad} quality bytes differ from the oracle ({ref['kind']})"
        assert cb.bed_text(out["events"], ref["names"]) == ref["bed"]
        assert out["counters"] == ref["counters"]
    m.close(); bb.close()


def test_gpu_shard_phases_by_hand():
    """the three shard phases driven from Python in the worst order a scheduler could pick: every begin first, then the carries from
    left to right, then the ends from right to left"""
    data, bb, batch, mask = dataset("c1s")
    args = ["-1"]
    ref = run_oracle(data, args)
    n_sh = 4
    shards, end = cb.plan_region_shards(batch, n_sh)
    subs = [cb.sub_batch(batch, sh["h0"], sh["r1"]) for sh in shards]
    ctxs = [cb.Crumble(params_from_args(args), device=0) for _ in range(n_sh)]
    for k, sh in enumerate(shards):
        ctxs[k].shard_begin(subs[k][0], cb.shard_window(sh))
    carry = None
    for k, sh in enumerate(shards):
        carry = ctxs[k].shard_carry(carry if sh["first"] != 1 else None, want_out=sh["hi_tid"] >= 0)
    outs = [None] * n_sh
    for k in reversed(range(n_sh)):
        outs[k] = ctxs[k].shard_end()
    n = int(batch.n_reads); off = bb.offsets()
    qual = np.zeros(int(batch.qual_bytes), np.uint8); done = np.zeros(n, bool)
    cnt = {k: 0 for k in cb.COUNTER_NAMES}; evs = []
    for k, sh in enumerate(shards):
        fin = cb.shard_final_mask(batch, sh, end, done)
        idx = np.arange(sh["h0"], sh["r1"])[fin]; base = int(off[sh["h0"]])
        for i in idx:
            q0 = int(off[i]); q1 = int(off[i + 1]) if i + 1 < n else int(batch.qual_bytes)
            qual[q0:q1] = outs[k]["qual"][q0 - base: q1 - base]
        done[idx] = True
        for c in cnt: cnt[c] += outs[k]["counters"][c]
        evs.append(outs[k]["events"])
    assert done.all()
    assert int((qual[mask] != ref["qual"][mask]).sum()) == 0
    assert cb.bed_text(np.concatenate(evs), ref["names"]) == ref["bed"] and cnt == ref["counters"]
    for g in ctxs: g.close()


@pytest.mark.parametrize("tag", ["plain", "t", "T", "efg", "EFGt", "all"])
def test_gpu_cli_aux_tag_options(tag):
    """-t / -T / -e..-G (purge_tags, snp_score.c:989-1054) through the crumble_gpu command line on the GPU: whole SAM output vs the
    reference's, for reads with i, Z, A, f, H and B-array tags"""
    from test_host import TAGS
    cli = ROOT / "crumble_b200" / "lib" / "crumble_gpu"
    with tempfile.TemporaryDirectory() as td:
        out = os.path.join(td, "o.sam")
        r = subprocess.run([str(cli), "-z"] + TAGS[tag] + [str(GDIR / "tags.sam"), out], stderr=subprocess.PIPE, text=True)
        assert r.returncode == 0, r.stderr
        assert open(out).read() == open(GDIR / f"tags.{tag}.out.sam").read()


def test_gpu_very_deep_columns():
    """columns deeper than MAX_DEPTH = 20000 (snp_score.c:92, 1493-1500): VDEEP BED lines, counted but unprocessed columns; one call,
    streamed in small chunks, chained through the command line, and over region shards"""
    data, nr, nb = cb.simulate("C4", 0.01, seed=9, amplicon_depth=16000, n_amplicons=2, threads=2)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish(pack=True); m = valid_mask(bb)
    for args in (["-9"], ["-1"]):
        ref = run_oracle(data, args)
        assert ref["bed"].count("VDEEP") >= 50
        g = cb.Crumble(params_from_args(args), device=0)
        g.set_chunk_bytes(1 << 20)
        out = g.process(batch)
        assert int((out["qual"][m] != ref["qual"][m]).sum()) == 0
        assert cb.bed_text(out["events"], ref["names"]) == ref["bed"] and out["counters"] == ref["counters"]
        g.close()
        mm = cb.MultiCrumble(params_from_args(args), devices=[0, 0, 0])
        out = mm.process(batch)
        assert int((out["qual"][m] != ref["qual"][m]).sum()) == 0
        assert cb.bed_text(out["events"], ref["names"]) == ref["bed"] and out["counters"] == ref["counters"]
        mm.close()
        r = run_oracle(data, args, binary=ROOT / "crumble_b200" / "lib" / "crumble_gpu", kind="gpu-cli", env_extra={"CRUMBLE_BATCH_READS": "7000"})
        assert (r["qual"][m] == ref["qual"][m]).all() and r["bed"] == ref["bed"] and r["counters"] == ref["counters"]
    bb.close()
