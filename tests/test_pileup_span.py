"""A record's pileup span (cg_pileup_span, cg_core.h) and the "open at a cut" test (cg_open_at, cg_pipeline.h), against a plain model on
handmade records: every CIGAR op alone, ops that consume no reference, no CIGAR, placed unmapped and unplaced records, zero-length
reference ops, a contig change and a record of 65 535 ops.  The host sees the span through the batcher (cg_batch_ends, pmax_end,
cg_aligned_bases, cg_algorithmic_bytes), the device body through the emulated stream cut (cg_emu_stream_cut)."""
import ctypes as C

import numpy as np

import crumble_b200 as cb
from test_device_batch import host_dev_batch
from test_device_stream import model_cut, slib

REF_OPS = {0, 2, 3, 7, 8}          # M D N = X: the ops that consume the reference (SAM specification)


def model_span(tid, flag, ops):
    """rule 1: 0 outside the pileup (unplaced, unmapped, no op consumes the reference), else the reference span, at least 1"""
    if tid < 0 or flag & 4 or not any(op in REF_OPS for _, op in ops):
        return 0
    return max(sum(n for n, op in ops if op in REF_OPS), 1)


def records():
    """(tid, pos, flag, [(len, op)], l_qseq), sorted by (tid, pos) with the unplaced ones last"""
    r = [(0, 100 + 2 * op, 0, [(10 + op, op)], 10) for op in range(10)]           # each op 0-9 alone
    r += [
        (0, 130, 0, [(3, 1), (4, 4), (2, 5), (1, 6)], 7),                            # I S H P: no reference op
        (0, 131, 0, [], 12),                                                          # n_cigar = 0
        (0, 132, 4, [(50, 0)], 50),                                                   # flag 4 on a placed record
        (0, 133, 0, [(40, 2)], 0),                                                    # D only
        (0, 134, 0, [(3000, 3)], 0),                                                  # N only: open across every later cut of the contig
        (0, 140, 0, [(0, 0), (5, 4)], 5),                                             # a zero-length M: span 1
        (0, 141, 0, [(0, 2), (4, 1)], 4),                                             # a zero-length D: span 1
        (0, 141, 0, [(10, 0)], 10),
        (0, 142, 0, [(10, 0)], 10),
        (0, 150, 0, [(1, 0 if k % 2 == 0 else 1) for k in range(65535)], 65535),     # 65 535 ops: 32 768 M, 32 767 I
        (0, 160, 0, [(5, 4), (20, 0), (7, 2), (20, 8), (3, 3), (20, 7), (5, 4)], 50),
        (1, 5, 0, [(20, 0)], 20),                                                     # contig change below the last end of contig 0
        (1, 6, 4, [], 10),
        (1, 8, 0, [(15, 2), (5, 0)], 5),
        (1, 9, 0, [(5, 0)], 5),
        (1, 30, 0, [(5, 0)], 5),
        (-1, -1, 0, [(30, 0)], 30),                                                   # tid = -1 with a reference op
        (-1, -1, 4, [], 8),
    ]
    return r


def build(recs):
    rng = np.random.default_rng(11)
    bb = cb.BatchBuilder(pinned=False)
    for tid, pos, flag, ops, l in recs:
        cig = np.array([(n << 4) | op for n, op in ops], np.uint32)
        bb.add(tid, pos, flag, 60, cig, rng.integers(0, 256, (l + 1) // 2, dtype=np.uint8), rng.integers(2, 41, l, dtype=np.uint8))
    return bb, bb.finish()


def test_host_span_end_and_sums():
    recs = records()
    bb, batch = build(recs)
    tid = np.array([r[0] for r in recs]); pos = np.array([r[1] for r in recs], np.int64)
    span = np.array([model_span(t, fl, ops) for t, _, fl, ops, _ in recs], np.int64)
    assert span[10 + 9] == 32768 and list(span[:10]) == [10, 0, 12, 13, 0, 0, 0, 17, 18, 0]
    end = pos + span
    assert np.array_equal(cb.batch_ends(batch), end)
    pmax = end.copy()
    for i in range(1, len(recs)):
        if tid[i] == tid[i - 1]:
            pmax[i] = max(pmax[i - 1], end[i])
    assert np.array_equal(np.ctypeslib.as_array(batch.pmax_end, shape=(len(recs),)), pmax)
    pile = span > 0
    ln = np.array([r[4] for r in recs], np.int64); nc = np.array([len(r[3]) for r in recs], np.int64)
    assert cb.aligned_bases(batch) == int(ln[pile].sum())
    assert cb.algorithmic_bytes(batch) == int(((ln + 1) // 2 + 2 * ln + 4 * nc + 16)[pile].sum())
    bb.close()


def test_device_span_at_cuts():
    """the stream cut of every prefix of the records (k_prep_read's and k_stream_plan's bodies): S and f as the model of the two rules
    predicts them"""
    recs = records()
    bb, batch = build(recs)
    f = cb.concat_fields(batch)
    span = [model_span(t, fl, ops) for t, _, fl, ops, _ in recs]
    lib = slib()
    seen_open = False
    for k in range(1, len(recs) + 1):
        g = dict(f)
        ncig = int(f["n_cigar"][:k].astype(np.int64).sum())
        nq = int(f["l_qseq"][:k].astype(np.int64).sum())
        g.update({x: f[x][:k] for x in ("tid", "pos", "flag", "mapq", "l_qseq", "n_cigar")})
        g.update(cigar=f["cigar"][:ncig], qual=f["qual"][:nq], seq=f["seq"][: sum((int(l) + 1) // 2 for l in f["l_qseq"][:k])])
        for e0 in sorted({0, k // 2, k - 1}):
            for last in (0, 1):
                res = np.zeros(6, np.int32)
                lib.cg_emu_stream_cut(C.byref(host_dev_batch(g)), e0, last, res.ctypes.data)
                m, fx, hi_tid, X, S, skip = model_cut(list(g["tid"]), list(g["pos"]), list(g["flag"]), span[:k], e0, last)
                got = tuple(int(x) for x in res)
                assert (got[0], got[1], got[2], got[5]) == (m, fx, hi_tid, skip), (k, e0, last, got)
                if hi_tid >= 0:
                    assert (got[3], got[4]) == (X, S), (k, e0, last, got)
                    seen_open |= S < X
    assert seen_open
    bb.close()
