"""BASELINE.json's full-size configurations on the GPU against the CPU oracle at the SAME size (tests/util.py: the reference's own code
when oracle/_ref is built, else the restatement pinned to the stored vectors of tests/golden/oracle_runs.json):
synthetic chr20 (64 Mb at 30x: 1.29e7 reads, 1.92e9 aligned bases) at -9 (configs[1]) and -1 -B (configs[2]) over the whole file,
the 1 Mb region (configs[0]) and the 1000x amplicon panel (configs[3]); plus slicing invariance at full size."""
import numpy as np
import pytest

import crumble_b200 as cb
from util import header_names, run_oracle, valid_mask

pytestmark = pytest.mark.gpu


def _bytes_of(off, ln):
    """indices of the quality bytes of the given records (offset, length)"""
    tot = int(ln.sum())
    starts = np.repeat(off - np.concatenate(([0], np.cumsum(ln)[:-1])), ln)
    return starts + np.arange(tot, dtype=np.int64)


def _start_reference(fin, td, tag, args):
    """the oracle of record on the whole file, in the background: one core, about 75 s for chr20 at 30x"""
    import os, subprocess
    from util import oracle_bin
    binary, kind = oracle_bin()
    fout, fbed = os.path.join(td, f"out.{tag}.ubam"), os.path.join(td, f"out.{tag}.bed")
    pr = subprocess.Popen([str(binary), "-z", "-v"] + args + ["-b", fbed, "-O", "bam,raw", fin, fout], stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
    return pr, fout, fbed, kind, args


def _collect_reference(pr, fout, fbed, kind, args, data_sha256):
    from util import parse_counters, pin_to_stored
    err = pr.communicate()[1]
    assert pr.returncode == 0, err[-2000:]
    out = np.fromfile(fout, dtype=np.uint8)
    rb = cb.BatchBuilder(pinned=False); rb.add_bam_stream(out); rb.finish()
    del out
    res = {"qual": rb.qual().copy(), "off": rb.offsets(), "len": rb.lengths(), "bed": open(fbed).read(), "counters": parse_counters(err), "kind": kind}
    pin_to_stored(res, data_sha256, args, valid_mask(rb))
    rb.close()
    return res


def test_full_size_c2_c3_whole_file_vs_reference():
    """BASELINE.json configs[1] (crumble -9) and configs[2] (crumble -1 -B) on the WHOLE synthetic chr20 (64 Mb, 30x: 1.29e7 reads,
    1.92e9 aligned bases): every quality byte, the BED text and the 19 counters of the GPU path against the reference's own code
    (or the pinned restatement) run over the whole file, one process per option set, while the GPU does its part; plus slicing invariance
    (resident == streamed at two chunk sizes) at this size."""
    import hashlib, os, tempfile
    data, n_reads, n_bases = cb.simulate("C2", 1.0, seed=2)
    data_sha256 = hashlib.sha256(data.tobytes()).hexdigest()
    assert n_reads > 12_000_000 and n_bases > 1_900_000_000
    names = header_names(data)
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        fin = os.path.join(td, "in.ubam"); data.tofile(fin)
        runs = {"C2": (["-9"], cb.default_params(9)), "C3": (["-1", "-B"], cb.default_params(1, binary_qual=1))}
        procs = {k: _start_reference(fin, td, k, a) for k, (a, _) in runs.items()}
        bb = cb.BatchBuilder()
        bb.add_bam_stream(data)
        del data
        batch = bb.finish()
        mask = valid_mask(bb)
        got = {}
        for k, (a, p) in runs.items():
            g = cb.Crumble(p, device=0)
            g.upload(batch); g.run()
            res = g.download(batch)
            ncols = g.n_columns()
            for chunk in ((96 << 20, 40 << 20) if k == "C2" else (64 << 20,)):
                g.set_chunk_bytes(chunk)
                o = g.process(batch)
                assert np.array_equal(o["qual"][mask], res["qual"][mask]), f"{k}: streamed ({chunk >> 20} MiB chunks) differs from resident"
                assert o["counters"] == res["counters"] and len(o["events"]) == res["n_events"]
            if k == "C2":
                assert res["counters"]["columns"] == ncols              # every covered position is a counted column at -9
            got[k] = {"qual": o["qual"][mask].copy(), "bed": cb.bed_text(o["events"], names), "counters": o["counters"]}
            del o, res
            g.close()
        off, ln = bb.offsets(), bb.lengths()
        for k in runs:
            ref = _collect_reference(*procs[k], data_sha256)
            assert np.array_equal(ref["off"], off) and np.array_equal(ref["len"], ln), f"{k}: the reference wrote different records"
            nbad = int((got[k]["qual"] != ref["qual"][mask]).sum())
            assert nbad == 0, f"{k}: {nbad} of {int(mask.sum())} quality bytes differ from the reference run over the whole file"
            assert got[k]["bed"] == ref["bed"], f"{k}: BED text differs"
            assert got[k]["counters"] == ref["counters"], f"{k}: counters differ"
            if k == "C3":
                assert ref["counters"]["over_depth"] > 0 and ref["bed"].count("DEEP") > 0          # the sequential depth average is live at -1
        bb.close()


@pytest.mark.parametrize("preset,seed,args", [("C1", 1, ["-9"]), ("C4", 4, ["-9"]), ("C4", 4, ["-1"]), ("C1", 1, ["-1", "-B"])],
                         ids=lambda v: "".join(v) if isinstance(v, list) else str(v))
def test_full_size_c1_c4_exact(preset, seed, args):
    """BASELINE.json configs[0] (1 Mb at 30x) and configs[3] (1000x amplicon panel: hot columns, STR-rich, every read of an amplicon
    starting at the same column) at their full sizes, where the CPU oracle still finishes in seconds: bit-exact qualities, BED
    lines and counters, resident and streamed."""
    from test_gpu_parity import params_from_args
    data, n_reads, n_bases = cb.simulate(preset, 1.0, seed=seed)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    mask = valid_mask(bb)
    ref = run_oracle(data, args)
    g = cb.Crumble(params_from_args(args), device=0)
    g.set_chunk_bytes(8 << 20)
    out = g.process(batch)
    nbad = int((out["qual"][mask] != ref["qual"][mask]).sum())
    assert nbad == 0, f"{nbad} quality bytes differ from the oracle ({ref['kind']})"
    assert cb.bed_text(out["events"], ref["names"]) == ref["bed"]
    assert out["counters"] == ref["counters"]
    g.upload(batch); g.run(); res = g.download(batch)
    assert np.array_equal(res["qual"][mask], out["qual"][mask]) and res["counters"] == out["counters"]
    g.close(); bb.close()
