"""Read lengths other than 150 on the GPU: the three inputs of tests/test_read_lengths.py (nine simulated lengths merged, 100-base reads
with 161-168 and 177-350-base stretches, reads of 1 to 80 000 bases with many-op CIGARs and missing qualities) through every entry
point, against the pinned oracle: qualities, BED text and all 19 counters.  They reach both k_rewrite paths (blocks staged in shared
memory, at and just over the staging limit, and the thread-per-read fallback), its general path for reads longer than RW_GORIG, the
scalar form for 0xff and above -U bytes, and the per-record compact planes with many length codes as well as their plain-array
fallback (test_read_lengths.test_inputs_reach_every_rewrite_path asserts which)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import crumble_b200 as cb
from test_device_batch import params_from_opts
import test_read_lengths
from test_read_lengths import ARGS, INPUTS, dataset
from util import PORT_BIN, ROOT, run_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

CLI = ROOT / "crumble_b200" / "lib" / "crumble_gpu"
_refs = {}


def every(n, k):
    return list(range(k, n, k))


def oracle(name, args):
    """the pinned oracle's result for one input, computed once per process"""
    key = (name, tuple(args))
    if key not in _refs:
        _refs[key] = test_read_lengths.oracle(dataset(name)[0], args)
    return _refs[key]


def assert_oracle(out, ref, mask, what, host_layout=True):
    """host_layout: out["qual"] is the batch's padded buffer; otherwise the concatenated qualities of process_device / device_stream"""
    q = out["qual"][mask] if host_layout else out["qual"]
    nbad = int((q != ref["qual"][mask]).sum()) if q.size == int(mask.sum()) else -1
    assert nbad == 0, f"{what}: {nbad} quality bytes differ from the oracle ({ref['kind']})"
    assert cb.bed_text(out["events"], ref["names"]) == ref["bed"], what
    assert out["counters"] == ref["counters"], what


@pytest.mark.parametrize("args", ARGS, ids=lambda a: "".join(a))
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_host_batch_entry_points(name, args):
    """cg_process resident and in 64 KB upload chunks (slices cut through the long reads), upload / run / download, the packed batch
    (compact per-record planes, or the plain arrays where the batch does not qualify), region shards on 3 and 5 contexts, and the
    multi-device scheduler on 3 contexts"""
    data, bb, batch, mask = dataset(name)
    ref = oracle(name, args)
    p = params_from_opts(args)
    g = cb.Crumble(p, device=0)
    assert_oracle(g.process(batch), ref, mask, "resident")
    g.set_chunk_bytes(1 << 16)
    assert_oracle(g.process(batch), ref, mask, "64 KB chunks")
    g.upload(batch); g.run()
    assert_oracle(g.download(batch), ref, mask, "upload / run / download")
    pb = cb.BatchBuilder(); pb.add_bam_stream(data); packed = pb.finish(pack=True)
    assert packed.meta_planes == (0 if name == "long" else 1)
    g.set_chunk_bytes(0)
    assert_oracle(g.process(packed), ref, mask, "packed")
    g.upload(packed); g.run()
    assert_oracle(g.download(packed), ref, mask, "packed, upload / run / download")
    for n_sh in (3, 5):
        ctxs = [cb.Crumble(p, device=0) for _ in range(n_sh)]
        assert_oracle(cb.run_region_shards(ctxs, batch, n_sh), ref, mask, f"{n_sh} region shards")
        for c in ctxs:
            c.close()
    m = cb.MultiCrumble(p, devices=[0] * 3)
    for b, what in ((batch, "plain"), (packed, "packed")):
        assert_oracle(m.process(b), ref, mask, f"multi-device scheduler, {what}")
    m.close(); g.close(); pb.close()


@pytest.mark.parametrize("args", [["-9"], ["-1", "-B"], ["-3", "-U35", "-Y0.2"]], ids=lambda a: "".join(a))
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_device_entry_points(name, args):
    """process_device into a new tensor and in place, and device_stream cut every 7 (not on the long-read input) and 97 records and
    at seeded random cuts"""
    data, bb, batch, mask = dataset(name)
    ref = oracle(name, args)
    g = cb.Crumble(params_from_opts(args), device=0)
    t = cb.device_batch(batch, 0)
    r = g.process_device(t)
    assert_oracle(dict(r, qual=r["qual"].cpu().numpy()), ref, mask, "process_device", host_layout=False)
    t2 = {k: v.clone() for k, v in t.items()}
    r = g.process_device(t2, out=t2["qual"])
    assert r["qual"].data_ptr() == t2["qual"].data_ptr()
    assert_oracle(dict(r, qual=t2["qual"].cpu().numpy()), ref, mask, "process_device in place", host_layout=False)
    n = int(batch.n_reads)
    rng = np.random.default_rng(n)
    for cuts in ([] if name == "long" else [every(n, 7)]) + [every(n, 97), sorted(set(int(x) for x in rng.integers(0, n + 1, 40)))]:
        s = g.device_stream()
        q, ev, cnt = [], [], None
        for ch in cb.split_device_batch(t, cuts=cuts) + [None]:
            o = s.push(ch) if ch is not None else s.close()
            q.append(o["qual"].cpu().numpy()); ev.append(o["events"])
            cnt = o["counters"] if cnt is None else {k: cnt[k] + o["counters"][k] for k in cnt}
        assert_oracle({"qual": np.concatenate(q), "events": np.concatenate(ev), "counters": cnt}, ref, mask,
                      f"device_stream, cuts {cuts[:3]}...", host_layout=False)
    g.close()


@pytest.mark.parametrize("name", ["boundary", "mixed"])
def test_device_stream_every_record(name):
    """device_stream with one record per push for the first 1000 records (every cut falls inside the reach of the reads before
    it), the rest in one push"""
    data, bb, batch, mask = dataset(name)
    ref = oracle(name, ["-9"])
    g = cb.Crumble(params_from_opts(["-9"]), device=0)
    s = g.device_stream()
    q, ev, cnt = [], [], None
    for ch in cb.split_device_batch(cb.device_batch(batch, 0), cuts=list(range(1, 1001))) + [None]:
        o = s.push(ch) if ch is not None else s.close()
        q.append(o["qual"].cpu().numpy()); ev.append(o["events"])
        cnt = o["counters"] if cnt is None else {k: cnt[k] + o["counters"][k] for k in cnt}
    assert_oracle({"qual": np.concatenate(q), "events": np.concatenate(ev), "counters": cnt}, ref, mask, "one record per push", host_layout=False)
    g.close()


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_chained_calls(name):
    """the crumble_gpu command line cut every 7 (not on the long-read input), 211 and 5000 records"""
    data, bb, batch, mask = dataset(name)
    for args in (["-9"], ["-1"]):
        ref = oracle(name, args)
        for reads in ((211, 5000) if name == "long" else (7, 211, 5000)):
            r = run_oracle(data, args, binary=CLI, kind="gpu-cli", env_extra={"CRUMBLE_BATCH_READS": str(reads)})
            nbad = int((r["qual"][mask] != ref["qual"][mask]).sum())
            assert nbad == 0 and r["bed"] == ref["bed"] and r["counters"] == ref["counters"], (args, reads, nbad)


def test_columns_bit_exact_mixed_lengths():
    """per-column consensus and decisions on the mixed-length input at -9, every field bit for bit (discrep included), against the
    oracle's column dump"""
    data, bb, batch, mask = dataset("mixed")
    g = cb.Crumble(params_from_opts(["-9"]), device=0)
    cols = g.process(batch, want_columns=True)["columns"]
    g.close()
    with tempfile.TemporaryDirectory() as td:
        fin, dump = os.path.join(td, "i.ubam"), os.path.join(td, "cols.bin")
        data.tofile(fin)
        subprocess.run([str(PORT_BIN), "-z", "-9", fin, "mem:x"], check=True, env=dict(os.environ, ORACLE_COLUMN_DUMP=dump))
        exp = np.fromfile(dump, dtype=cb.api.COLUMN_DTYPE)
    assert len(cols) == len(exp) > 50000
    for f in ("tid", "pos", "n_plp", "call", "het_call", "phred", "het_phred"):
        assert np.array_equal(cols[f], exp[f]), f
    assert np.array_equal(cols["discrep"].view(np.uint32), exp["discrep"].view(np.uint32)), "discrep differs bitwise"
    for bit, nm in ((1, "preserve"), (2, "keep_qual"), (4, "window active"), (8, "processed")):
        assert np.array_equal(cols["flags"] & bit, exp["flags"] & bit), nm
    assert np.array_equal((cols["flags"] >> 8) & 31, (exp["flags"] >> 8) & 31), "BED tags"
