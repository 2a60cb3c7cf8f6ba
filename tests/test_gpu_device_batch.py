"""cg_process_device on the GPU: records already in GPU memory (torch tensors of concatenated BAM fields) in, rewritten qualities in GPU
memory out.  Against the oracle on tiny at every level, and against cg_process on the same context in the same run (qualities after
stripping, BED, the 19 counters and the column dump bit-exact) on the parity data sets, the STR-at-depth, ambiguity-code, VDEEP and
edge-case inputs and the options served by the plain per-item kernels; at full size; in stream order; in place; interleaved with
cg_process; and with inputs it must reject."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import crumble_b200 as cb
from crumble_b200.api import DevBatch, Result
from test_device_batch import params_from_opts, sam_batch
from test_gpu_parity import LEVELS, dataset
from test_oracle import EDGE, GDIR, GOLD
from util import add_ambiguity_codes, run_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def strip(batch, padded):
    """the qualities of a cg_process result (batch layout) back to back, as cg_process_device lays them out"""
    b = cb.api.Batch.from_buffer_copy(batch)
    b.qual = np.ascontiguousarray(padded).ctypes.data_as(C.POINTER(C.c_uint8))
    return cb.concat_fields(b)["qual"]


def both(g, batch, want_columns=True):
    """cg_process then cg_process_device on the same context"""
    ref = g.process(batch, want_columns=want_columns)
    ref["qual"] = strip(batch, ref["qual"])
    dev = g.process_device(cb.device_batch(batch, g.device), want_columns=want_columns)
    torch.cuda.synchronize()
    dev["qual"] = dev["qual"].cpu().numpy()
    return ref, dev


def assert_same(ref, dev, what=""):
    nbad = int((ref["qual"] != dev["qual"]).sum()) if ref["qual"].size == dev["qual"].size else -1
    assert nbad == 0, f"{what}: {nbad} quality bytes differ"
    assert np.array_equal(ref["events"], dev["events"]), what
    assert ref["counters"] == dev["counters"], what
    if "columns" in ref:
        assert ref["columns"].tobytes() == dev["columns"].tobytes(), what


def check_same(batch, args, names=("chr1", "chr2")):
    g = cb.Crumble(params_from_opts(args, names), device=0)
    ref, dev = both(g, batch)
    assert_same(ref, dev, " ".join(args))
    assert g.h2d_bytes() == 0
    g.close()


@pytest.mark.parametrize("args", LEVELS, ids=lambda a: "".join(a))
def test_tiny_all_levels_against_oracle(args):
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_opts(args), device=0)
    out = g.process_device(cb.device_batch(batch, 0))
    q = out["qual"].cpu().numpy()
    ref = run_oracle(data, args)
    assert int((q != ref["qual"][mask]).sum()) == 0, f"quality bytes differ from the oracle ({ref['kind']})"
    assert cb.bed_text(out["events"], ref["names"]) == ref["bed"]
    assert out["counters"] == ref["counters"]
    g.close()


@pytest.mark.parametrize("name", ["c1s", "c2s", "c4s", "c4m"])
@pytest.mark.parametrize("args", [["-9"], ["-1", "-B"], ["-5"]], ids=lambda a: "".join(a))
def test_equals_process(name, args):
    check_same(dataset(name)[2], args)


@pytest.mark.parametrize("name,args", [("c4m", ["-9", "-D300"]), ("c4m", ["-1", "-D300", "-X0.2"]), ("c4s", ["-1", "-D300", "-Q300"])],
                         ids=lambda v: "".join(v) if isinstance(v, list) else v)
def test_str_triggers_at_depth(name, args):
    check_same(dataset(name)[2], args)


@pytest.mark.parametrize("name,rate", [("tiny", 0.01), ("c4s", 0.002), ("c1s", 0.05)])
def test_ambiguity_codes(name, rate):
    data, n = add_ambiguity_codes(dataset(name)[0], rate, seed=7)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    for args in (["-9"], ["-1", "-B"], ["-3"]):
        check_same(batch, args)
    bb.close()


def test_very_deep_columns():
    data, nr, nb = cb.simulate("C4", 0.01, seed=9, amplicon_depth=16000, n_amplicons=2, threads=2)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    for args in (["-9"], ["-1"]):
        check_same(batch, args)
    bb.close()


@pytest.mark.parametrize("tag", sorted(EDGE))
def test_edge_cases(tag):
    bb, names = sam_batch(GDIR / "edge_cases.sam", pinned=True)
    check_same(bb.finish(), EDGE[tag], names)
    bb.close()


OPT_ARGS = [a for a in sorted(GOLD["tiny"]["opt_runs"]) if "-y" not in a]


@pytest.mark.parametrize("args", OPT_ARGS + ["-9 -r chr1:20000-40000", "-1 -r chr2:1000-30000"], ids=lambda a: a.replace(" ", ""))
def test_options(args):
    """-k/-K/-N/-S/-R keep.bed (the plain per-item kernels) and -r"""
    check_same(dataset("tiny")[2], [str(GDIR / "keep.tiny.bed") if x == "BED" else x for x in args.split()])


@pytest.mark.parametrize("args", [["-9"], ["-1", "-B"]], ids=lambda a: "".join(a))
def test_full_size(args):
    """whole synthetic chr20 (C2, -9) and C3 (-1 -B): same quality bytes as cg_process, nothing copied to the device from the host"""
    preset = "C2" if args == ["-9"] else "C3"
    data, nr, nb = cb.simulate(preset, 1.0, seed=100)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    del data
    g = cb.Crumble(params_from_opts(args, ["chr20"]), device=0)
    ref = g.process(batch)
    ref_sha = hashlib.sha256(strip(batch, ref["qual"]).tobytes()).hexdigest()
    t = cb.device_batch(batch, 0)
    out = g.process_device(t)
    assert g.h2d_bytes() == 0
    assert hashlib.sha256(out["qual"].cpu().numpy().tobytes()).hexdigest() == ref_sha
    assert np.array_equal(out["events"], ref["events"]) and out["counters"] == ref["counters"]
    g.close(); bb.close()


def test_stream_order():
    """input made by a torch kernel on a non-default stream (held back behind a long sleep), the call, and a torch kernel consuming
    the result, all queued on that stream with no synchronisation by the caller in between"""
    data, bb, batch, mask = dataset("c1s")
    g = cb.Crumble(params_from_opts(["-1"]), device=0)
    ref, _ = both(g, batch, want_columns=False)
    t = cb.device_batch(batch, 0)
    key = torch.tensor(0x5a, dtype=torch.uint8, device="cuda")
    scrambled = t["qual"] ^ key
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
        t2 = dict(t, qual=scrambled ^ key)                       # the real qualities exist only once this kernel has run
        out = g.process_device(t2)
        consumed = (out["qual"].to(torch.int32) + 1).to(torch.int64)
    s.synchronize()
    assert np.array_equal(consumed.cpu().numpy() - 1, ref["qual"].astype(np.int64))
    assert np.array_equal(out["events"], ref["events"]) and out["counters"] == ref["counters"]
    g.close()


def test_inputs_unchanged_and_in_place():
    data, bb, batch, mask = dataset("c2s")
    g = cb.Crumble(params_from_opts(["-9"]), device=0)
    t = cb.device_batch(batch, 0)
    keep = {k: v.clone() for k, v in t.items()}
    a = g.process_device(t)
    torch.cuda.synchronize()
    for k in t:
        assert torch.equal(t[k], keep[k]), f"{k} changed"
    b = g.process_device(t, out=t["qual"])
    assert b["qual"].data_ptr() == t["qual"].data_ptr()
    assert torch.equal(a["qual"], t["qual"]) and np.array_equal(a["events"], b["events"]) and a["counters"] == b["counters"]
    g.close()


def test_context_state_across_calls():
    """one context: calls of different sizes alternate and cg_process interleaves with cg_process_device; every result equals its own
    reference from a fresh context"""
    refs = {}
    for name in ("tiny", "c1s", "c4s"):
        g = cb.Crumble(params_from_opts(["-5"]), device=0)
        refs[name] = both(g, dataset(name)[2], want_columns=False)[0]
        g.close()
    g = cb.Crumble(params_from_opts(["-5"]), device=0)
    for name, how in (("c1s", "dev"), ("tiny", "host"), ("tiny", "dev"), ("c4s", "dev"), ("c1s", "host"), ("c1s", "dev"), ("tiny", "dev")):
        batch = dataset(name)[2]
        if how == "dev":
            r = g.process_device(cb.device_batch(batch, 0))
            r["qual"] = r["qual"].cpu().numpy()
        else:
            r = g.process(batch)
            r["qual"] = strip(batch, r["qual"])
        assert_same(refs[name], r, f"{name} {how}")
    g.close()


def test_events_refetched_not_rerun():
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_opts(["-1"]), device=0)
    ref, _ = both(g, batch, want_columns=False)
    assert len(ref["events"]) > 1
    g2 = cb.Crumble(params_from_opts(["-1"]), device=0)
    t = cb.device_batch(batch, 0)
    out = g2.process_device(t, out=t["qual"], events_cap=1)           # in place: a second run would rewrite rewritten qualities
    assert np.array_equal(out["events"], ref["events"]) and out["counters"] == ref["counters"]
    assert np.array_equal(out["qual"].cpu().numpy(), ref["qual"])
    g.close(); g2.close()


def test_rejected_inputs_leave_the_context_usable():
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_opts(["-9"]), device=0)
    good = g.process_device(cb.device_batch(batch, 0))
    good_q = good["qual"].cpu().numpy()
    t = cb.device_batch(batch, 0)
    bad = [dict(t, pos=t["pos"].cpu()),                                  # a CPU tensor
           dict(t, tid=t["tid"].to(torch.int64)),                        # a wrong dtype
           dict(t, mapq=t["mapq"][:-1]),                                 # a length mismatch
           dict(t, qual=t["qual"][:-1])]                                 # qual_len != sum of l_qseq (found on the device)
    if torch.cuda.device_count() > 1:
        bad.append(dict(t, cigar=t["cigar"].to("cuda:1")))              # memory of another device
    for k, b in enumerate(bad):
        with pytest.raises(cb.CrumbleError):
            g.process_device(b)
        r = g.process_device(t)
        assert np.array_equal(r["qual"].cpu().numpy(), good_q) and r["counters"] == good["counters"], k
    # the C entry on its own: a host pointer, and a device pointer of another device, are not device memory of the context's device
    lib = cb.load_lib()
    host = np.zeros(int(t["tid"].numel()), np.int32)
    db = DevBatch(n_reads=t["tid"].numel(), n_cigar_total=t["cigar"].numel(), seq_len=t["seq"].numel(), qual_len=t["qual"].numel())
    for k in cb.api.DEV_FIELDS:
        setattr(db, k, t[k].data_ptr())
    db.tid = host.ctypes.data
    res = Result()
    assert lib.cg_process_device(g.h, C.byref(db), C.c_void_p(t["qual"].data_ptr()), C.byref(res)) == -4
    assert b"not device memory" in lib.cg_last_error(g.h)
    if torch.cuda.device_count() > 1:
        other = t["tid"].to("cuda:1")
        db.tid = other.data_ptr()
        assert lib.cg_process_device(g.h, C.byref(db), C.c_void_p(t["qual"].data_ptr()), C.byref(res)) == -4
    r = g.process_device(t)
    assert np.array_equal(r["qual"].cpu().numpy(), good_q)
    g.close()
