"""CPU tests of the device-resident entry (cg_process_device): the numpy half of ``device_batch`` (stripping a host batch into
concatenated BAM fields), and the ingest / emit bodies of k_ingest / k_emit (cg_pipeline.h) run by the host emulation
(tests/emu/libcg_emu.so), whose cg_process_device must give what its cg_process gives on the same records."""
import ctypes as C
import re

import numpy as np
import pytest

import crumble_b200 as cb
from crumble_b200.api import Batch, BedEvent, BedReg, Column, COLUMN_DTYPE, DevBatch, EVENT_DTYPE, Result
from test_oracle import EDGE, GDIR, GOLD, sim
from util import ROOT

EMU_LIB = ROOT / "tests" / "emu" / "libcg_emu.so"
NT16 = "=ACMGRSVTWYHKDBN"


# ---- shared with tests/test_gpu_device_batch.py ------------------------------------------------------------------------------------
def params_from_opts(args, names=("chr1", "chr2")):
    """cg_params for a crumble option list: levels, the numeric options, -k/-K, -N, -S, -R <bed file> and -r <contig:beg-end>"""
    p = cb.default_params()
    lib = cb.load_lib()
    it = iter(args)
    for a in it:
        k, v = a[1], a[2:]
        if k in "YqQUmCZPpLDXkKRr" and not v:
            v = next(it)
        if k in "135789": lib.cg_params_level(C.byref(p), int(k))
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
        elif k == "N": p.perfect_col = 1
        elif k == "S": p.softclip = 1
        elif k in "kK":
            for q in v.split(","):
                lo, _, hi = q.partition("-")
                for x in range(int(lo), int(hi or lo) + 1):
                    p.preserve_qual[x] = 1 + (k == "K")
        elif k == "R":
            regs = sorted((names.index(f[0]), int(f[1]), int(f[2])) for f in (l.split() for l in open(v)) if f and not f[0].startswith("#"))
            arr = (BedReg * len(regs))(*[BedReg(*r) for r in regs])
            p.bed, p.nbed = C.cast(arr, C.POINTER(BedReg)), len(regs)
            p._keep_bed = arr
        elif k == "r":
            m = re.fullmatch(r"(\w+):(\d+)-(\d+)", v)
            p.region_tid, p.region_beg, p.region_end = names.index(m[1]), int(m[2]) - 1, int(m[3])
        else:
            raise ValueError(a)
    return p


def sam_batch(path, pinned=False):
    """BatchBuilder of the records of a SAM file (SEQ '*' = no bases, QUAL '*' = 0xff), and the contig names"""
    names, bb = [], cb.BatchBuilder(pinned=pinned)
    for line in open(path):
        f = line.rstrip("\n").split("\t")
        if line.startswith("@"):
            if f[0] == "@SQ":
                names.append(dict(x.split(":", 1) for x in f[1:])["SN"])
            continue
        cig = [] if f[5] == "*" else [(int(n) << 4) | "MIDNSHP=X".index(op) for n, op in re.findall(r"(\d+)([MIDNSHP=X])", f[5])]
        seq = "" if f[9] == "*" else f[9].upper()
        codes = [NT16.index(c) for c in seq] + [0] * (len(seq) & 1)
        seq4 = np.array([(codes[i] << 4) | codes[i + 1] for i in range(0, len(codes), 2)], np.uint8)
        qual = np.full(len(seq), 255, np.uint8) if f[10] == "*" else np.frombuffer(f[10].encode(), np.uint8) - 33
        bb.add(names.index(f[2]) if f[2] != "*" else -1, int(f[3]) - 1, int(f[1]), int(f[4]), np.array(cig, np.uint32), seq4, qual[: len(seq)])
    return bb, names


def random_batch(seed, n=400, pinned=False):
    """records of random lengths (0, 1, odd, even, long), random bases including the phantom nibble of odd lengths, random CIGARs"""
    rng = np.random.default_rng(seed)
    bb = cb.BatchBuilder(pinned=pinned)
    pos = 0
    for i in range(n):
        l = int(rng.choice([0, 1, 2, 3, 7, 8, 9, 15, 16, 17, 100, 101, 150, 151, 599]) if rng.random() < 0.5 else rng.integers(0, 320))
        pos += int(rng.integers(0, 5))
        cig = np.array([(l << 4) | 0] if l and rng.random() < 0.7 else [(int(rng.integers(1, 50)) << 4) | int(rng.integers(0, 9)) for _ in range(int(rng.integers(0, 6)))], np.uint32)
        bb.add(0, pos, 0, 60, cig, rng.integers(0, 256, (l + 1) // 2, dtype=np.uint8), rng.integers(0, 94, l, dtype=np.uint8))
    return bb


# ---- the numpy half of device_batch ---------------------------------------------------------------------------------------------------
def expected_fields(batch):
    n = int(batch.n_reads)
    get = lambda ptr, cnt: np.ctypeslib.as_array(ptr, shape=(cnt,)) if cnt else np.zeros(0, np.uint8)
    off, ln = get(batch.off, n), get(batch.l_qseq, n)
    coff, nc = get(batch.cigar_off, n), get(batch.n_cigar, n)
    qual, seq, cig = get(batch.qual, int(batch.qual_bytes)), get(batch.seq, int(batch.seq_bytes)), get(batch.cigar, int(batch.n_cigar_total))
    return (np.concatenate([qual[o:o + l] for o, l in zip(off, ln)] + [np.zeros(0, np.uint8)]),
            np.concatenate([seq[o // 2:o // 2 + (l + 1) // 2] for o, l in zip(off, ln)] + [np.zeros(0, np.uint8)]),
            np.concatenate([cig[c:c + k] for c, k in zip(coff, nc)] + [np.zeros(0, np.uint32)]))


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_concat_fields_round_trip(seed):
    """stripping the batcher's padding: qualities, sequences (ceil(l/2) bytes, phantom nibble kept) and CIGARs of every record at its
    Batch.off / cigar_off, back to back; the row-mask path of a packed batch and the index path of a caller's own layout agree"""
    bb = random_batch(seed)
    batch = bb.finish()
    q, s, c = expected_fields(batch)
    ln = bb.lengths()
    assert (ln == 0).any() and (ln == 1).any() and (ln % 2 == 1).any() and ((ln % 2 == 0) & (ln > 0)).any()
    for b in (batch, Batch.from_buffer_copy(batch)):
        if b is not batch:
            b.packed = 0
        f = cb.concat_fields(b)
        assert np.array_equal(f["qual"], q) and np.array_equal(f["seq"], s) and np.array_equal(f["cigar"], c)
        assert f["qual"].size == ln.sum() and f["seq"].size == ((ln + 1) // 2).sum()
        assert np.array_equal(f["l_qseq"], ln) and f["tid"].dtype == np.int32 and f["flag"].dtype == np.uint16 and f["cigar"].dtype == np.uint32
    bb.close()


def test_concat_fields_empty_batch():
    f = cb.concat_fields(cb.BatchBuilder(pinned=False).finish())
    assert all(v.size == 0 for v in f.values())


# ---- the emulated cg_process_device ---------------------------------------------------------------------------------------------------
_emu = None


def emu():
    global _emu
    if _emu is None:
        lib = C.CDLL(str(EMU_LIB))
        lib.cg_create.restype = C.c_void_p
        lib.cg_create.argtypes = [C.POINTER(cb.Params), C.c_int, C.POINTER(C.c_int)]
        lib.cg_destroy.argtypes = [C.c_void_p]
        lib.cg_last_error.restype = C.c_char_p
        lib.cg_last_error.argtypes = [C.c_void_p]
        lib.cg_process.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Result)]
        lib.cg_process_device.argtypes = [C.c_void_p, C.POINTER(DevBatch), C.c_void_p, C.POINTER(Result)]
        lib.cg_emu_ingest.restype = C.c_int64
        lib.cg_emu_ingest.argtypes = [C.POINTER(DevBatch), C.c_void_p, C.c_void_p]
        _emu = lib
    return _emu


def host_dev_batch(f):
    """a cg_dev_batch over numpy arrays: the emulation's "device" memory is host memory"""
    db = DevBatch(n_reads=f["tid"].size, n_cigar_total=f["cigar"].size, seq_len=f["seq"].size, qual_len=f["qual"].size)
    for k in cb.api.DEV_FIELDS:
        setattr(db, k, f[k].ctypes.data if f[k].size else None)
    return db


def emu_result(events_cap, columns_cap):
    ev, cols = np.zeros(events_cap, EVENT_DTYPE), np.zeros(max(columns_cap, 1), COLUMN_DTYPE)
    res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=events_cap,
                 columns=cols.ctypes.data_as(C.POINTER(Column)), columns_cap=max(columns_cap, 1))
    return res, ev, cols


def emu_call(p, fn):
    lib = emu()
    err = C.c_int(0)
    ctx = lib.cg_create(C.byref(p), 0, C.byref(err))
    assert ctx, err.value
    try:
        return fn(lib, ctx)
    finally:
        lib.cg_destroy(ctx)


def emu_reference(p, batch):
    """emulated cg_process: stripped qualities, events, counters, column dump"""
    def run(lib, ctx):
        n_cols = 1
        for _ in range(2):
            res, ev, cols = emu_result(1 << 16, n_cols)
            qout = np.zeros(max(int(batch.qual_bytes), 1), np.uint8)
            res.qual_out = qout.ctypes.data_as(C.POINTER(C.c_uint8))
            assert lib.cg_process(ctx, C.byref(batch), C.byref(res)) == 0, lib.cg_last_error(ctx)
            if res.n_columns <= n_cols:
                break
            n_cols = int(res.n_columns)
        b = Batch.from_buffer_copy(batch); b.qual = qout.ctypes.data_as(C.POINTER(C.c_uint8))
        return {"qual": cb.concat_fields(b)["qual"], "events": ev[: int(res.n_events)].copy(), "counters": list(res.counters),
                "columns": cols[: int(res.n_columns)].copy()}
    return emu_call(p, run)


def emu_device(p, f, in_place=False, columns_cap=1 << 16):
    def run(lib, ctx):
        db = host_dev_batch(f)
        out = f["qual"] if in_place else np.full(f["qual"].size, 0xab, np.uint8)
        res, ev, cols = emu_result(1 << 16, columns_cap)
        e = lib.cg_process_device(ctx, C.byref(db), out.ctypes.data if out.size else None, C.byref(res))
        assert e == 0, lib.cg_last_error(ctx)
        return {"qual": out, "events": ev[: int(res.n_events)].copy(), "counters": list(res.counters), "columns": cols[: int(res.n_columns)].copy()}
    return emu_call(p, run)


def assert_same(a, b):
    assert np.array_equal(a["qual"], b["qual"]), f"{int((a['qual'] != b['qual']).sum())} quality bytes differ"
    assert np.array_equal(a["events"], b["events"]) and a["counters"] == b["counters"]
    assert len(a["columns"]) == len(b["columns"]) and a["columns"].tobytes() == b["columns"].tobytes()


@pytest.mark.parametrize("seed", [4, 5])
def test_emulated_ingest_builds_the_batchers_layout(seed):
    """k_ingest's body on concatenated fields gives back the batcher's padded arrays byte for byte: qualities at off, sequences at off/2,
    zero padding in both, the phantom low nibble of odd-length records"""
    tiny = cb.BatchBuilder(pinned=False)
    tiny.add_bam_stream(sim("tiny"))
    for bb in (random_batch(seed), tiny):
        batch = bb.finish()
        f = cb.concat_fields(batch)
        db = host_dev_batch(f)
        padded = emu().cg_emu_ingest(C.byref(db), None, None)
        assert padded == int(batch.qual_bytes)
        q, s = np.full(padded, 0xee, np.uint8), np.full(padded // 2, 0xee, np.uint8)
        emu().cg_emu_ingest(C.byref(db), q.ctypes.data, s.ctypes.data)
        assert np.array_equal(q, bb.qual()) and np.array_equal(s, np.ctypeslib.as_array(batch.seq, shape=(int(batch.seq_bytes),)))
        bb.close()


EMU_ARGS = [["-9"], ["-1", "-B"], ["-5", "-q30"], ["-3", "-P1.5"]]


@pytest.mark.parametrize("name", sorted(GOLD))
@pytest.mark.parametrize("args", EMU_ARGS, ids=lambda a: "".join(a))
def test_emulated_process_device_equals_process(name, args):
    """golden data sets: cg_process_device on the concatenated fields equals cg_process on the batch (qualities compared after
    stripping), events, counters and column dump included"""
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(sim(name)); batch = bb.finish()
    p = params_from_opts(args)
    ref = emu_reference(p, batch)
    assert_same(emu_device(p, cb.concat_fields(batch), columns_cap=len(ref["columns"])), ref)
    bb.close()


@pytest.mark.parametrize("tag", sorted(EDGE))
def test_emulated_process_device_edge_cases(tag):
    """zero-length (SEQ '*'), single-base, odd-length, unmapped, no-reference-op and clipped records and the trailing tid = -1 records"""
    bb, names = sam_batch(GDIR / "edge_cases.sam")
    batch = bb.finish()
    assert (bb.lengths() == 0).any() and (bb.lengths() % 2 == 1).any() and (np.ctypeslib.as_array(batch.tid, shape=(int(batch.n_reads),))[-3:] == -1).all()
    p = params_from_opts(EDGE[tag], names)
    ref = emu_reference(p, batch)
    assert_same(emu_device(p, cb.concat_fields(batch), columns_cap=len(ref["columns"])), ref)


def test_emulated_process_device_in_place_and_options():
    """the rewrite in place (qual_out = the input qualities) and the options served by the plain per-item bodies"""
    bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(sim("tiny")); batch = bb.finish()
    for args in (["-9"], ["-1", "-R", str(GDIR / "keep.tiny.bed"), "-p", "8"], ["-5", "-S", "-K", "37", "-N"], ["-9", "-K", "11", "-k", "25"]):
        p = params_from_opts(args)
        ref = emu_reference(p, batch)
        f = cb.concat_fields(batch)
        assert_same(emu_device(p, f, in_place=True, columns_cap=len(ref["columns"])), ref)


def test_emulated_process_device_rejects_inconsistent_sums():
    bb = random_batch(7, n=50); batch = bb.finish()
    f = cb.concat_fields(batch)
    p = params_from_opts(["-9"])

    def run(lib, ctx):
        out = np.zeros(f["qual"].size, np.uint8)
        for field, delta in (("qual_len", -1), ("seq_len", 1), ("n_cigar_total", -1)):
            db = host_dev_batch(f)
            setattr(db, field, getattr(db, field) + delta)
            res, _, _ = emu_result(16, 0)
            assert lib.cg_process_device(ctx, C.byref(db), out.ctypes.data, C.byref(res)) == -4
            assert b"sums disagree" in lib.cg_last_error(ctx)
        neg = dict(f, l_qseq=f["l_qseq"].copy())
        neg["l_qseq"][3] = -neg["l_qseq"][3] - 1
        res, _, _ = emu_result(16, 0)
        assert lib.cg_process_device(ctx, C.byref(host_dev_batch(neg)), out.ctypes.data, C.byref(res)) == -4
        res, _, _ = emu_result(16, 0)
        assert lib.cg_process_device(ctx, C.byref(host_dev_batch(f)), out.ctypes.data, C.byref(res)) == 0    # still usable
        return 0
    emu_call(p, run)
