"""CPU tests of streams of device records (cg_stream_device), run by the host emulation (tests/emu/libcg_emu.so) with the plan / cut /
keep / retain / ingest / emit bodies of cg_device.cu's kernels around the emulated window chain: a stream cut anywhere gives what one
cg_process_device on the whole batch gives (qualities in stream order, concatenated events, summed counters), the cut model, the edge
cases and the rejections."""
import ctypes as C

import numpy as np
import pytest

import crumble_b200 as cb
from crumble_b200.api import BedEvent, DevBatch, EVENT_DTYPE, Result, StreamOut
from test_device_batch import emu_device, host_dev_batch, params_from_opts, sam_batch
from test_oracle import EDGE, GDIR, GOLD, sim
from util import ROOT

STREAM_LIB = ROOT / "tests" / "emu" / "libcg_emu_stream.so"
CG_ERR_BAD_ARG, CG_ERR_UNSORTED, CG_ERR_STATE = -4, -5, -8
_slib = None


def slib():
    """the emulation with the stream entry (tests/emu/stream.mk); the references come from libcg_emu.so (emu_device)"""
    global _slib
    if _slib is None:
        lib = C.CDLL(str(STREAM_LIB))
        lib.cg_create.restype = C.c_void_p
        lib.cg_create.argtypes = [C.POINTER(cb.Params), C.c_int, C.POINTER(C.c_int)]
        lib.cg_destroy.argtypes = [C.c_void_p]
        lib.cg_last_error.restype = C.c_char_p
        lib.cg_last_error.argtypes = [C.c_void_p]
        lib.cg_process.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.cg_process_device.argtypes = [C.c_void_p, C.POINTER(DevBatch), C.c_void_p, C.POINTER(Result)]
        lib.cg_stream_device.argtypes = [C.c_void_p, C.POINTER(DevBatch), C.c_int, C.c_void_p, C.c_int64, C.POINTER(Result), C.POINTER(StreamOut)]
        lib.cg_emu_stream_cut.argtypes = [C.POINTER(DevBatch), C.c_int64, C.c_int, C.c_void_p]
        lib.cg_process_window.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.cg_download.argtypes = [C.c_void_p, C.POINTER(Result)]
        _slib = lib
    return _slib


def emu_call(p, fn):
    """fn(lib, ctx) on a fresh context of the stream emulation"""
    lib = slib()
    err = C.c_int(0)
    ctx = lib.cg_create(C.byref(p), 0, C.byref(err))
    assert ctx, err.value
    try:
        return fn(lib, ctx)
    finally:
        lib.cg_destroy(ctx)


def push(lib, ctx, chunk, held_qual, last=False, events_cap=1 << 16, qual_cap=None, alias=False):
    """one call; returns (code, emitted qualities, events, counters, StreamOut)"""
    db = host_dev_batch(chunk) if chunk is not None else None
    new = chunk["qual"].size if chunk is not None else 0
    cap = held_qual + new if qual_cap is None else qual_cap
    out = chunk["qual"] if alias else np.full(max(cap, 1), 0xab, np.uint8)
    ev = np.zeros(events_cap, EVENT_DTYPE)
    res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=events_cap)
    so = StreamOut()
    code = lib.cg_stream_device(ctx, C.byref(db) if db is not None else None, int(last), out.ctypes.data if out.size else None, cap, C.byref(res), C.byref(so))
    if code == 0 and res.n_events > events_cap:              # fetched again, not run again
        ev = np.zeros(int(res.n_events), EVENT_DTYPE)
        res2 = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=int(res.n_events))
        assert lib.cg_download(ctx, C.byref(res2)) == 0
        res = res2
    return code, out[: int(so.qual_len)].copy(), ev[: int(res.n_events)].copy(), list(res.counters), so


def run_stream(lib, ctx, chunks, close_empty=False, events_cap=1 << 16, alias=False):
    """push every chunk (the last one with last = 1, or an empty close after it); the concatenated result and the held counts"""
    q, ev, cnt, held, held_q, nrec = [], [], np.zeros(19, np.int64), [], 0, 0
    for i, ch in enumerate(chunks):
        last = i == len(chunks) - 1 and not close_empty
        code, qq, ee, cc, so = push(lib, ctx, ch, held_q, last=last, events_cap=events_cap, alias=alias)
        assert code == 0, lib.cg_last_error(ctx)
        assert qq.size == so.qual_len and so.n_records >= 0
        q.append(qq); ev.append(ee); cnt += cc; held.append(int(so.held_records)); held_q = int(so.held_qual_len); nrec += int(so.n_records)
    if close_empty:
        code, qq, ee, cc, so = push(lib, ctx, None, held_q, last=True, events_cap=events_cap)
        assert code == 0, lib.cg_last_error(ctx)
        q.append(qq); ev.append(ee); cnt += cc; nrec += int(so.n_records); held.append(int(so.held_records))
    assert held[-1] == 0
    return {"qual": np.concatenate(q), "events": np.concatenate(ev), "counters": [int(x) for x in cnt], "n_records": nrec, "held": held}


def stream_emu(p, f, chunks, **kw):
    return emu_call(p, lambda lib, ctx: run_stream(slib(), ctx, chunks, **kw))


def check_stream(p, f, ref, cuts, **kw):
    chunks = cb.split_device_batch(f, cuts=cuts)
    got = stream_emu(p, f, chunks, **kw)
    n = f["tid"].size
    assert got["n_records"] == n
    bad = int((got["qual"] != ref["qual"]).sum()) if got["qual"].size == ref["qual"].size else -1
    assert bad == 0, f"{bad} quality bytes differ"
    assert np.array_equal(got["events"], ref["events"]), "events differ"
    assert got["counters"] == [int(x) for x in ref["counters"]], "counters differ"
    return got


_data = {}


def dataset(name):
    if name not in _data:
        bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(sim(name)); batch = bb.finish()
        _data[name] = (bb, batch, cb.concat_fields(batch))
    return _data[name][2]


def every(n, k):
    return list(range(k, n, k))


def random_cuts(n, seed, k=12):
    rng = np.random.default_rng(seed)
    return sorted(set(int(x) for x in rng.integers(0, n + 1, k)))


STREAM_ARGS = [["-9"], ["-1"], ["-3"], ["-5", "-q30"], ["-1", "-m10", "-C0.05", "-Z0.01"], ["-3", "-i0.5,3", "-s2.0,1"]]


def args_params(args):
    """params_from_opts plus -i / -s (STR multiplier, addend)"""
    rest, p_over = [], {}
    for a in args:
        if a[1] in "is":
            mul, add = a[2:].split(",")
            p_over[f"{a[1]}STR_mul"], p_over[f"{a[1]}STR_add"] = float(mul), int(add)
        else:
            rest.append(a)
    p = params_from_opts(rest)
    for k, v in p_over.items():
        setattr(p, k, v)
    return p


@pytest.mark.parametrize("name", sorted(GOLD))
@pytest.mark.parametrize("args", STREAM_ARGS, ids=lambda a: "".join(a))
def test_stream_equals_whole_batch(name, args):
    """cut every 7, 97, 1500 and 20000 records and at seeded random cuts: the emitted qualities concatenated, the events concatenated
    and the counters summed equal the emulated cg_process_device on the whole batch"""
    f = dataset(name)
    p = args_params(args)
    ref = emu_device(p, f, columns_cap=0)
    n = f["tid"].size
    for k in (7, 97, 1500, 20000):
        check_stream(p, f, ref, every(n, k))
    for seed in (1, 2):
        check_stream(p, f, ref, random_cuts(n, seed + len(name)))


@pytest.mark.parametrize("name", sorted(GOLD))
@pytest.mark.parametrize("args", STREAM_ARGS, ids=lambda a: "".join(a))
def test_stream_one_record_per_push(name, args):
    """the smallest chunks: every record on its own, the last one closed by an empty call"""
    f = dataset(name)
    p = args_params(args)
    ref = emu_device(p, f, columns_cap=0)
    got = check_stream(p, f, ref, every(f["tid"].size, 1), close_empty=True)
    assert max(got["held"]) < 2000


OPT_ARGS = [a for a in sorted(GOLD["tiny"]["opt_runs"]) if "-y" not in a]


@pytest.mark.parametrize("args", OPT_ARGS, ids=lambda a: a.replace(" ", ""))
def test_stream_options(args):
    """-k/-K/-N/-S/-R keep.bed (the plain per-item bodies) at 211 records per push"""
    f = dataset("tiny")
    p = params_from_opts([str(GDIR / "keep.tiny.bed") if x == "BED" else x for x in args.split()])
    ref = emu_device(p, f, columns_cap=0)
    check_stream(p, f, ref, every(f["tid"].size, 211))


@pytest.mark.parametrize("tag", sorted(t for t in EDGE if "-r" not in EDGE[t]))
@pytest.mark.parametrize("k", [1, 5, 40])
def test_stream_edge_cases(tag, k):
    """zero-length, single-base, odd-length, unmapped, no-reference-op and clipped records, and the trailing unplaced ones"""
    bb, names = sam_batch(GDIR / "edge_cases.sam")
    batch = bb.finish()
    f = cb.concat_fields(batch)
    p = params_from_opts(EDGE[tag], names)
    ref = emu_device(p, f, columns_cap=0)
    check_stream(p, f, ref, every(f["tid"].size, k))
    check_stream(p, f, ref, every(f["tid"].size, k), close_empty=True)


def synthetic(records):
    """a concatenated-fields dict from (tid, pos, flag, cigar ops [(len, op)], length) tuples"""
    rng = np.random.default_rng(5)
    f = {k: [] for k in ("tid", "pos", "flag", "mapq", "l_qseq", "n_cigar", "cigar", "seq", "qual")}
    for tid, pos, flag, cig, l in records:
        f["tid"].append(tid); f["pos"].append(pos); f["flag"].append(flag); f["mapq"].append(60); f["l_qseq"].append(l)
        f["n_cigar"].append(len(cig)); f["cigar"] += [(n << 4) | "MIDNSHP=X".index(o) for n, o in cig]
        f["seq"] += list(rng.choice([0x11, 0x12, 0x24, 0x48, 0x84, 0x21], (l + 1) // 2))
        f["qual"] += list(rng.integers(2, 41, l))
    return {k: np.array(v, dtype=cb.api.DEV_FIELDS[k]) for k, v in f.items()}


def test_stream_contigs_unplaced_mates_and_shared_keys():
    """both contigs of tiny with a cut right at the contig change; placed unmapped mates right behind an open read; a tail of unplaced
    records; a push whose records all share one key (everything held, nothing emitted); empty pushes in between"""
    f = dataset("tiny")
    n = f["tid"].size
    p = params_from_opts(["-9"])
    ref = emu_device(p, f, columns_cap=0)
    change = int(np.argmax(f["tid"] != f["tid"][0]))
    assert 0 < change < n
    check_stream(p, f, ref, [change - 1, change, change + 1])
    recs = []
    for i in range(60):
        recs.append((0, 100 + 3 * i, 0, [(100, "M")], 100))
        if i % 7 == 0:
            recs += [(0, 100 + 3 * i, 4, [], 100), (0, 100 + 3 * i, 4, [], 100)]    # placed unmapped mates, same key as the read
    recs += [(0, 400, 0, [(50, "M"), (5000, "D"), (50, "M")], 100)]                    # a long open read
    recs += [(0, 401, 4, [], 90)] * 5 + [(0, 402 + i, 0, [(100, "M")], 100) for i in range(30)]
    recs += [(0, 500, 0, [(80, "M")], 80)] * 25                                           # one key
    recs += [(-1, -1, 4, [], 70)] * 9                                                    # unplaced tail
    g = synthetic(recs)
    m = g["tid"].size
    for args in (["-9"], ["-1"]):
        p = params_from_opts(args)
        ref = emu_device(p, g, columns_cap=0)
        for cuts in (every(m, 1), every(m, 3), [m - 40, m - 30, m - 20, m - 9], random_cuts(m, 3, 20)):
            check_stream(p, g, ref, cuts)
        same = int(np.argmax((g["pos"] == 500)))
        chunks = cb.split_device_batch(g, cuts=[same, same + 25, same + 25])
        empty = {k: v[:0] for k, v in g.items()}

        def run(lib, ctx):
            lib = slib()
            code, q0, _, _, so0 = push(lib, ctx, chunks[0], 0)
            assert code == 0
            code, q1, e1, c1, so1 = push(lib, ctx, chunks[1], int(so0.held_qual_len))
            assert code == 0 and so1.n_records == 0 and q1.size == 0 and so1.held_records >= 25     # all behind the long open read
            code, q2, _, _, so2 = push(lib, ctx, empty, int(so1.held_qual_len))
            assert code == 0 and so2.n_records == 0 and so2.held_records == so1.held_records
            code, q3, _, _, so3 = push(lib, ctx, None, int(so2.held_qual_len))
            assert code == 0 and so3.n_records == 0
            code, q4, _, _, so4 = push(lib, ctx, chunks[3], int(so3.held_qual_len), last=True)
            assert code == 0 and so4.held_records == 0
            return np.concatenate([q0, q1, q2, q3, q4])
        assert np.array_equal(emu_call(p, run), ref["qual"])


def test_close_with_nothing_held():
    f = dataset("tiny")
    p = params_from_opts(["-9"])

    def run(lib, ctx):
        lib = slib()
        code, q, e, c, so = push(lib, ctx, None, 0, last=True)            # a stream that never got a record
        assert code == 0 and q.size == 0 and so.n_records == 0 and so.held_records == 0 and not any(c)
        ch = cb.split_device_batch(f, cuts=[100])[0]
        code, q, e, c, so = push(lib, ctx, ch, 0)
        assert code == 0
        while ch["tid"][-1] != -1 and so.held_records:                    # flush with last = 1 on an empty push
            code, q2, e, c, so = push(lib, ctx, None, int(so.held_qual_len), last=True)
            assert code == 0 and so.held_records == 0
        code, q3, e, c, so = push(lib, ctx, None, 0, last=True)
        assert code == 0 and so.n_records == 0
        return 0
    emu_call(p, run)


def test_aliased_output_and_small_event_buffer():
    """qual_out = the chunk's own qualities (everything is ingested before anything is emitted), and events_cap = 1 (fetched again)"""
    f = dataset("c1s")
    p = params_from_opts(["-1"])
    ref = emu_device(p, f, columns_cap=0)
    n = f["tid"].size
    got = stream_emu(p, f, cb.split_device_batch(f, cuts=every(n, 3000)), events_cap=1)
    assert np.array_equal(got["qual"], ref["qual"]) and np.array_equal(got["events"], ref["events"])

    def run(lib, ctx):
        lib = slib()
        q = []
        for i, c in enumerate(cb.split_device_batch(f, cuts=every(n, 3000))):
            buf = np.zeros(c["qual"].size + (4 << 20), np.uint8); buf[: c["qual"].size] = c["qual"]     # room for the held bytes too
            c = dict(c, qual=buf[: c["qual"].size])
            db = host_dev_batch(c)
            ev = np.zeros(1 << 16, EVENT_DTYPE)
            res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=1 << 16)
            so = StreamOut()
            last = i == len(range(3000, n, 3000))
            assert lib.cg_stream_device(ctx, C.byref(db), int(last), buf.ctypes.data, buf.size, C.byref(res), C.byref(so)) == 0
            q.append(buf[: int(so.qual_len)].copy())
        return np.concatenate(q)
    assert np.array_equal(emu_call(p, run), ref["qual"])


def model_cut(tid, pos, flag, span, e0, last):
    """the cut of DESIGN.md §3.6 in plain Python: m, f, hi_tid, X, S"""
    n = len(tid)
    pile = [t >= 0 and not (fl & 4) and s > 0 for t, fl, s in zip(tid, flag, span)]
    m, hi_tid, X = n, -1, 0
    if not last and n and tid[-1] >= 0:
        key = (tid[-1], pos[-1])
        m = 1 + max([i for i in range(n) if (tid[i], pos[i]) != key], default=-1)
        if m > 0 and tid[m - 1] == tid[-1]:
            hi_tid, X = tid[-1], pos[-1]
    S = X
    if hi_tid >= 0:
        S = min([pos[i] for i in range(m) if pile[i] and tid[i] == hi_tid and pos[i] + span[i] > X] + [X])
    f = m
    if hi_tid >= 0:
        f = min([i for i in range(e0, m) if pile[i] and tid[i] == hi_tid and pos[i] + span[i] > X] + [m])
    skip = m <= e0
    if skip:
        f = e0
    return m, f, hi_tid, X, S, int(skip)


@pytest.mark.parametrize("seed", range(6))
def test_cut_model(seed):
    """k_stream_plan's per-record body and the cut from its reductions, against the plain model, on random sorted streams with shared
    keys, unmapped mates, reads without reference operations, contig changes and unplaced tails"""
    rng = np.random.default_rng(seed)
    lib = slib()
    for trial in range(40):
        n = int(rng.integers(1, 60))
        recs, tid, pos = [], 0, int(rng.integers(0, 50))
        for i in range(n):
            u = rng.random()
            if u < 0.05:
                tid += 1; pos = int(rng.integers(0, 30))
            elif u < 0.5:
                pos += int(rng.integers(0, 4))
            if rng.random() < 0.03 and i > n // 2:
                recs += [(-1, -1, 4, [], 10)] * (n - i)
                break
            kind = rng.random()
            if kind < 0.15:
                recs.append((tid, pos, 4, [], 10))
            elif kind < 0.2:
                recs.append((tid, pos, 0, [(10, "S")], 10))
            else:
                recs.append((tid, pos, 0, [(int(rng.integers(1, 30)), "M")] + ([(int(rng.integers(1, 40)), "D"), (5, "M")] if rng.random() < 0.2 else []), 10))
        g = synthetic(recs)
        span = [sum(x >> 4 for x in g["cigar"][sum(g["n_cigar"][:i]):sum(g["n_cigar"][:i + 1])] if (x & 15) in (0, 2, 3, 7, 8)) for i in range(len(recs))]
        span = [max(s, 1) if any((x & 15) in (0, 2, 3, 7, 8) for x in g["cigar"][sum(g["n_cigar"][:i]):sum(g["n_cigar"][:i + 1])]) else 0 for i, s in enumerate(span)]
        for last in (0, 1):
            e0 = int(rng.integers(0, len(recs) + 1))
            res = np.zeros(6, np.int32)
            lib.cg_emu_stream_cut(C.byref(host_dev_batch(g)), e0, last, res.ctypes.data)
            exp = model_cut(list(g["tid"]), list(g["pos"]), list(g["flag"]), span, e0, last)
            m, f, hi_tid, X, S, skip = exp
            got = tuple(int(x) for x in res)
            assert got[0] == m and got[1] == f and got[2] == hi_tid and got[5] == skip, (trial, got, exp)
            if hi_tid >= 0:
                assert got[3] == X and got[4] == S, (trial, got, exp)


def test_rejections_leave_the_stream_unchanged():
    """qual_cap one byte short, a -r region, a column dump: CG_ERR_BAD_ARG and the stream goes on as if the call had not been made; other
    compute calls while the stream is open: CG_ERR_STATE; a chunk that breaks the sort order: CG_ERR_UNSORTED, and a fresh stream on the
    same context then succeeds"""
    f = dataset("c1s")
    n = f["tid"].size
    p = params_from_opts(["-9"])
    ref = emu_device(p, f, columns_cap=0)
    chunks = cb.split_device_batch(f, cuts=every(n, 997))

    def run(lib, ctx):
        lib = slib()
        q, held_q = [], 0
        for i, ch in enumerate(chunks):
            last = i == len(chunks) - 1
            code, *_ = push(lib, ctx, ch, held_q, last=last, qual_cap=held_q + ch["qual"].size - 1)
            assert code == CG_ERR_BAD_ARG
            ev = np.zeros(4, EVENT_DTYPE); cols = np.zeros(4, cb.api.COLUMN_DTYPE)
            res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=4, columns=cols.ctypes.data_as(C.POINTER(cb.api.Column)), columns_cap=4)
            out = np.zeros(held_q + ch["qual"].size + 1, np.uint8)
            assert lib.cg_stream_device(ctx, C.byref(host_dev_batch(ch)), 0, out.ctypes.data, out.size, C.byref(res), C.byref(StreamOut())) == CG_ERR_BAD_ARG
            if i == 1:
                res = Result()
                assert lib.cg_process_device(ctx, C.byref(host_dev_batch(ch)), out.ctypes.data, C.byref(res)) == CG_ERR_STATE
                assert lib.cg_process(ctx, None, C.byref(res)) == CG_ERR_STATE
                assert lib.cg_process_window(ctx, None, None, C.byref(res)) == CG_ERR_STATE
            code, qq, _, _, so = push(lib, ctx, ch, held_q, last=last)
            assert code == 0
            q.append(qq); held_q = int(so.held_qual_len)
        assert np.array_equal(np.concatenate(q), ref["qual"])
        # unsorted across chunks: the second chunk starts before the first one ends
        a, b = cb.split_device_batch(f, cuts=[3000])[0], cb.split_device_batch(f, cuts=[1000, 2000])[1]
        code, _, _, _, so = push(lib, ctx, a, 0)
        assert code == 0
        code, *_ = push(lib, ctx, b, int(so.held_qual_len))
        assert code == CG_ERR_UNSORTED
        got = run_stream(lib, ctx, chunks)                                # a fresh stream: the failed one was closed
        assert np.array_equal(got["qual"], ref["qual"])
        return 0
    emu_call(p, run)
    pr = params_from_opts(["-9", "-r", "chr1:20000-40000"])

    def run_r(lib, ctx):
        code, *_ = push(slib(), ctx, chunks[0], 0)
        assert code == CG_ERR_BAD_ARG
        return 0
    emu_call(pr, run_r)


def test_split_device_batch_views():
    """the chunks are consecutive, cover every record and field once, and empty chunks come out where cuts repeat"""
    f = dataset("c1s")
    n = f["tid"].size
    cuts = [0, 5, 5, 1234, n]
    ch = cb.split_device_batch(f, cuts=cuts)
    assert len(ch) == len(cuts) + 1 and ch[0]["tid"].size == 0 and ch[2]["tid"].size == 0 and ch[-1]["tid"].size == 0
    for k in f:
        assert np.array_equal(np.concatenate([c[k] for c in ch]), f[k])
    assert sum(c["tid"].size for c in cb.split_device_batch(f, 1000)) == n
    with pytest.raises(cb.CrumbleError):
        cb.split_device_batch(f)
