"""Read lengths other than 150 on the CPU: the emulated pipeline (tests/emu/emu_crumble) against the pinned oracle on three seeded
inputs, uncut, cut into chained calls and spread over emulated devices.

The inputs are built here, bit-identically from their seeds, and are shared with tests/test_gpu_read_lengths.py:
  mixed_stream     tiny at nine read lengths (60 to 400) merged into one coordinate-sorted stream;
  boundary_stream  100-base reads with a few 177-350-base reads carrying indels, and one stretch of 161-168-base reads that fills a
                   k_rewrite block of 128 records to exactly its staging limit;
  long_read_stream reads of 1 to 20 000 bases and a few longer than 65 535, CIGARs of 1 to several hundred ops (M = X I D N S H P),
                   missing ('*') qualities, qualities up to 93, more than 256 distinct lengths.
rewrite_paths() mirrors the block range rule of k_rewrite (crumble_b200/csrc/cg_device.cu) so that the tests can assert which of its
paths the inputs reach; a change to a generator that stops reaching one fails here instead of quietly testing less.

The oracle's vectors for these inputs are stored in tests/golden/oracle_runs.read_lengths.json (same format as oracle_runs.json);
oracle() pins every run to them.  To re-record: CRUMBLE_ORACLE_RECORD=runs.jsonl pytest tests/test_read_lengths.py, then write the
recorded lines into that file, one vector per line."""
import bisect
import hashlib
import struct

import numpy as np
import pytest

import crumble_b200 as cb
import util
from util import EMU_BIN, ROOT, run_oracle, valid_mask

LENGTH_RUNS = ROOT / "tests" / "golden" / "oracle_runs.read_lengths.json"


def oracle(data, args):
    """run_oracle, pinned (or recorded) to the stored vectors of these inputs in LENGTH_RUNS instead of oracle_runs.json"""
    stored = util.STORED
    util.STORED = LENGTH_RUNS
    try:
        return run_oracle(data, args)
    finally:
        util.STORED = stored


# ---- uncompressed BAM streams ---------------------------------------------------------------------------------------------------------
CIGAR_OPS = "MIDNSHP=X"
NT4 = np.array([1, 2, 4, 8], np.uint8)                            # A C G T as nt16


def split_stream(data):
    """header bytes and [(tid, pos, record bytes)] of an uncompressed BAM stream"""
    b = data.tobytes()
    p = 8 + struct.unpack_from("<i", b, 4)[0]
    n = struct.unpack_from("<i", b, p)[0]; p += 4
    for _ in range(n):
        p += 4 + struct.unpack_from("<i", b, p)[0] + 4
    hdr, recs = b[:p], []
    while p + 4 <= len(b):
        bs = struct.unpack_from("<i", b, p)[0]
        tid, pos = struct.unpack_from("<ii", b, p + 4)
        recs.append((tid, pos, b[p:p + 4 + bs])); p += 4 + bs
    return hdr, recs


def bam_header(contigs):
    text = "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in contigs).encode()
    out = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(contigs))
    for n, l in contigs:
        out += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", l)
    return out


def reg2bin(beg, end):
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def bam_record(name, tid, pos, flag, mapq, cigar, bases, qual):
    """cigar [(op, len)], bases nt16 codes (uint8 array), qual uint8 array (0xff = '*')"""
    span = sum(n for op, n in cigar if op in "MDN=X")
    nm = name.encode() + b"\0"
    codes = np.append(bases, np.zeros(len(bases) & 1, np.uint8))
    seq = ((codes[0::2] << 4) | codes[1::2]).astype(np.uint8).tobytes()
    core = struct.pack("<iiBBHHHiiii", tid, pos, len(nm), mapq, reg2bin(max(pos, 0), max(pos, 0) + max(span, 1)), len(cigar), flag,
                       len(bases), -1, -1, 0)
    body = core + nm + b"".join(struct.pack("<I", (n << 4) | CIGAR_OPS.index(op)) for op, n in cigar) + seq + qual.astype(np.uint8).tobytes()
    return struct.pack("<i", len(body)) + body


def merge_streams(streams, fractions, seed):
    """a seeded fraction of each stream's records on each contig (fractions[stream][tid]) and every unmapped one, sorted by
    (tid, pos, source, index), unmapped records last"""
    rng = np.random.default_rng(seed)
    hdr, allr = None, []
    for k, (data, f) in enumerate(zip(streams, fractions)):
        h, recs = split_stream(data)
        assert hdr is None or h == hdr, "streams with different headers"
        hdr = h
        keep = rng.random(len(recs)) < np.array([f[t] if t >= 0 else 1.0 for t, _, _ in recs])
        allr += [(t if t >= 0 else 1 << 30, p, k, i, x) for i, (t, p, x) in enumerate(recs) if t < 0 or keep[i]]
    allr.sort(key=lambda z: z[:4])
    return np.frombuffer(hdr + b"".join(z[4] for z in allr), np.uint8)


# ---- a synthetic genome and reads written here (simgen stops at 400 bases and one CIGAR shape) -------------------------------------
class Genome:
    """one random contig with planted STRs and shared SNP and indel sites; every site sits on haplotype 0, 1 or both"""

    def __init__(self, rng, length, n_snp, n_indel):
        self.ref = rng.integers(0, 4, length).astype(np.uint8)
        for p in range(500, length - 500, 2000):                 # STRs: unit of 1-4 bases, 5-15 copies
            u = rng.integers(0, 4, int(rng.integers(1, 5)))
            k = len(u) * int(rng.integers(5, 15))
            self.ref[p:p + k] = np.resize(u, k)
        self.snp = np.sort(rng.choice(np.arange(100, length - 100), n_snp, replace=False))
        self.snp_alt = ((self.ref[self.snp] + rng.integers(1, 4, n_snp)) % 4).astype(np.uint8)
        self.snp_hap = rng.integers(0, 3, n_snp)                  # 2 = both haplotypes
        near_str = np.arange(500, length - 500, 2000)[: n_indel // 2] + 3
        ind = np.unique(np.concatenate([near_str, rng.integers(100, length - 100, n_indel - len(near_str))]))
        self.indel = ind.tolist()
        self.indel_len = {int(p): int(rng.integers(-6, 7)) or 2 for p in ind}      # > 0 insertion, < 0 deletion
        self.indel_hap = {int(p): int(rng.integers(0, 3)) for p in ind}

    def read(self, rng, pos, L, n_events, clip=0.15):
        """(cigar, nt16 bases) of a mapped read of L query bases starting at pos, or None if it would run off the contig.  It carries
        the sites of its haplotype, 1 % errors and about n_events extra I / D / N / P ops between runs of M / = / X; ops never sit
        next to each other without an M-type run between them, and the read ends on an M-type op or a clip."""
        G = len(self.ref)
        hap = int(rng.integers(0, 2))
        cig, seq = [], []

        def add(op, n):
            if cig and cig[-1][0] == op:
                cig[-1][1] += n
            else:
                cig.append([op, n])

        if rng.random() < 0.05:
            add("H", int(rng.integers(1, 40)))
        head = int(rng.integers(1, L // 4 + 1)) if L >= 4 and rng.random() < clip else 0
        tail = int(rng.integers(1, L // 4 + 1)) if L >= 8 and rng.random() < clip else 0
        if head:
            add("S", head); seq.append(rng.integers(0, 4, head))
        body, q, rp = L - head - tail, 0, pos
        mean = max(body / (n_events + 1), 1.0)
        labels = ["M"] if n_events < 3 else ["M", "M", "=", "X"]
        while q < body:
            n = min(body - q, max(1, int(rng.geometric(1.0 / mean))))
            k = bisect.bisect_right(self.indel, rp)               # a shared indel site inside this run cuts it there
            site = self.indel[k] if k < len(self.indel) else -1
            if rp < site < rp + n and site - rp < body - q:
                n = site - rp
            else:
                site = -1
            if rp + n > G:
                return None
            s = self.ref[rp:rp + n].copy()
            a, b = np.searchsorted(self.snp, [rp, rp + n])
            on = (self.snp_hap[a:b] == 2) | (self.snp_hap[a:b] == hap)
            s[self.snp[a:b][on] - rp] = self.snp_alt[a:b][on]
            err = rng.random(n) < 0.01
            s[err] = (s[err] + 1) % 4
            add(labels[int(rng.integers(0, len(labels)))], n); seq.append(s)
            q += n; rp += n
            if q >= body:
                break
            if site >= 0 and self.indel_hap[site] in (2, hap):
                d = self.indel_len[site]
                if d > 0 and q + d < body:
                    add("I", d); seq.append(rng.integers(0, 4, d)); q += d
                elif d < 0:
                    add("D", -d); rp -= d
                continue
            if n_events and rng.random() < n_events / max(body / mean, 1):
                e = rng.random()
                if e < 0.4 and body - q > 8:
                    d = int(rng.integers(1, 8)); add("I", d); seq.append(rng.integers(0, 4, d)); q += d
                elif e < 0.8:
                    add("D", int(rng.integers(1, 8))); rp += cig[-1][1]
                elif e < 0.9:
                    add("N", int(rng.integers(50, 3000))); rp += cig[-1][1]
                else:
                    add("P", int(rng.integers(1, 4)))
        if tail:
            add("S", tail); seq.append(rng.integers(0, 4, tail))
        if rng.random() < 0.05:
            add("H", int(rng.integers(1, 40)))
        if rp > G:
            return None
        return [tuple(c) for c in cig], NT4[np.concatenate(seq)]


def python_stream(seed, length, n_snp, n_indel, draw):
    """records drawn by draw(rng, i) -> (pos, L, n_events) or None for a placed-unmapped record; sorted by position, ten unplaced
    records at the end.  Qualities 2-41, 5 % of reads 0-93, 2 % '*'."""
    rng = np.random.default_rng(seed)
    g = Genome(rng, length, n_snp, n_indel)
    recs, i = [], 0
    while True:
        d = draw(rng, i)
        if d is False:
            break
        i += 1
        mapq = int(rng.choice([60, 60, 60, 0, 3, 20, 255]))
        flag = int(rng.choice([0, 16, 99, 147, 1024 + 16]))
        if d is None:                                             # placed unmapped: no CIGAR, the mate's position
            L = int(rng.integers(1, 300)); pos = int(rng.integers(0, length))
            cig, bases, flag = [], NT4[rng.integers(0, 4, L)], 4 | 1 | 64
        else:
            pos, L, ne = d
            r = g.read(rng, pos, L, ne)
            if r is None:
                continue
            cig, bases = r
        L = len(bases)
        qual = rng.integers(2, 42, L) if rng.random() >= 0.05 else rng.integers(0, 94, L)
        if rng.random() < 0.02:
            qual = np.full(L, 0xff)
        recs.append((pos, len(recs), bam_record(f"r{i}", 0, pos, flag, mapq, cig, bases, qual)))
    recs.sort(key=lambda z: z[:2])
    tail = [bam_record(f"u{k}", -1, -1, 4, 0, [], NT4[rng.integers(0, 4, 50 + k)], rng.integers(2, 42, 50 + k)) for k in range(10)]
    return np.frombuffer(bam_header([("chrL", length)]) + b"".join(z[2] for z in recs) + b"".join(tail), np.uint8)


MIXED_LENGTHS = (60, 100, 151, 161, 168, 176, 177, 250, 400)


def mixed_stream(seed):
    """tiny (two 50 kb contigs, its own variants and planted features) simulated at nine read lengths and merged: on the first contig
    12 % of each (blocks of 128 records mostly fit the staging buffers), on the second mostly reads of 177 bases and more (mostly not)"""
    streams = [cb.simulate("tiny", 1.0, seed, threads=2, read_len=L)[0] for L in MIXED_LENGTHS]
    return merge_streams(streams, [(0.12, 0.3 if L >= 177 else 0.02) for L in MIXED_LENGTHS], seed)


def boundary_stream(seed):
    """40 kb at about 30x: 100-base reads, 5 % of reads of 177-350 bases with 1-4 indels; positions 16-24 kb hold 161-168-base
    reads (0.5 % of 177-350), so whole blocks of 128 records stage 128 x 168 quality bytes, and some just miss"""
    length, n = 40000, 12500

    def draw(rng, i):
        if i == n:
            return False
        if rng.random() < 0.01:
            return None
        pos = int(rng.integers(0, length - 400))
        stretch = 16000 <= pos < 24000
        if rng.random() < (0.005 if stretch else 0.05):
            return pos, int(rng.integers(177, 351)), int(rng.integers(1, 5))
        return pos, int(rng.integers(161, 169)) if stretch else 100, int(rng.random() < 0.1)
    return python_stream(seed, length, 60, 40, draw)


def long_read_stream(seed):
    """120 kb at about 20x: lengths log-uniform in 1-20 000 (and 1-400 for a quarter of the reads), three reads of 66-80 kb; a tenth
    of the reads up to 3000 bases have a dense CIGAR (up to a few hundred ops)"""
    length, n = 120000, 2000

    def draw(rng, i):
        if i == n:
            return False
        if rng.random() < 0.01:
            return None
        if i in (300, 1000, 1600):
            L = int(rng.integers(66000, 80000))
        elif rng.random() < 0.25:
            L = int(rng.integers(1, 401))
        else:
            L = int(np.exp(rng.uniform(0, np.log(20000)))) + 1
        pos = int(rng.integers(0, max(length - L - 1000, 1)))
        dense = L <= 3000 and rng.random() < 0.1
        return pos, L, int(L / rng.integers(8, 30)) if dense else int(rng.integers(0, 4))
    return python_stream(seed, length, 250, 90, draw)


INPUTS = {"mixed": (mixed_stream, 21), "boundary": (boundary_stream, 22), "long": (long_read_stream, 23)}
_inputs = {}


def dataset(name):
    """(data, BatchBuilder, batch, valid mask) of one input, built once per process"""
    if name not in _inputs:
        f, seed = INPUTS[name]
        data = f(seed)
        bb = cb.BatchBuilder(pinned=False)
        bb.add_bam_stream(data)
        batch = bb.finish()
        _inputs[name] = (data, bb, batch, valid_mask(bb))
    return _inputs[name]


# ---- which k_rewrite paths an input reaches -------------------------------------------------------------------------------------------
RW_READS, RW_QCAP, RW_CCAP, RW_GORIG = 128, 128 * 168, 3072, 176


def rewrite_paths(batch, qcap=35):
    """k_rewrite's block rule on a resident batch (blocks of 128 records from record 0): a block is staged when its quality range
    (from off / l_qseq, 16-aligned) is at most RW_QCAP + 16 bytes and its column range at most RW_CCAP + 16; otherwise every record in
    it takes the thread-per-read fallback.  The column range is bounded from above by the reference span of the block's pileup reads,
    so a block called staged here is staged on the device (the converse need not hold)."""
    n = int(batch.n_reads)
    arr = lambda p, cnt=n: np.ctypeslib.as_array(p, shape=(cnt,))
    off, ln = arr(batch.off).astype(np.int64), arr(batch.l_qseq).astype(np.int64)
    tid, pos, flag = arr(batch.tid), arr(batch.pos).astype(np.int64), arr(batch.flag)
    nc, co = arr(batch.n_cigar), arr(batch.cigar_off)
    cig = arr(batch.cigar, int(batch.n_cigar_total))
    qual = np.ctypeslib.as_array(batch.qual, shape=(int(batch.qual_bytes),))
    r = {"staged": 0, "fallback": 0, "staged_general_long": 0, "staged_simple_ff": 0, "staged_simple_above_U": 0, "max_staged_qbytes": 0,
         "min_fallback_qbytes": 1 << 62, "max_len": int(ln.max()), "max_ops": int(nc.max()), "distinct_lengths": len(np.unique(ln))}
    for b0 in range(0, n, RW_READS):
        s = slice(b0, min(b0 + RW_READS, n))
        L = ln[s]
        if not (L > 0).any():
            continue
        lo, hi = int(off[s][L > 0].min()), int((off[s] + L)[L > 0].max())
        qb = ((hi + 15) & ~15) - (lo & ~15)
        sb = ((((hi + 1) >> 1) + 15) & ~15) - ((lo >> 1) & ~15)
        mapped = (L > 0) & (tid[s] >= 0) & ((flag[s] & 4) == 0)
        spans = np.array([sum(int(c) >> 4 for c in cig[co[i]:co[i] + nc[i]] if (int(c) & 15) in (0, 2, 3, 7, 8)) for i in range(s.start, s.stop)])
        mapped &= spans > 0
        cols = int((pos[s] + spans)[mapped].max() - pos[s][mapped].min()) + 16 if mapped.any() else 0
        if qb > RW_QCAP + 16 or sb > RW_QCAP // 2 + 16:
            r["fallback"] += 1; r["min_fallback_qbytes"] = min(r["min_fallback_qbytes"], qb)
            continue
        if cols > RW_CCAP + 16:
            continue                                             # staged or not: the bound does not tell
        r["staged"] += 1; r["max_staged_qbytes"] = max(r["max_staged_qbytes"], qb)
        for i in np.nonzero(mapped)[0] + b0:
            c = cig[co[i]:co[i] + nc[i]]
            simple = nc[i] == 1 and (int(c[0]) & 15) in (0, 7, 8) and int(c[0]) >> 4 == ln[i]
            q = qual[off[i]:off[i] + ln[i]]
            if not simple and ln[i] > RW_GORIG:
                r["staged_general_long"] += 1
            if simple and (q == 0xff).all():
                r["staged_simple_ff"] += 1
            if simple and ((q > qcap) & (q < 0x80)).any():
                r["staged_simple_above_U"] += 1
    return r


def meta_planes(data):
    """(meta_planes, number of length codes) of the input packed as one batch (BatchBuilder.finish(pack=True))"""
    bb = cb.BatchBuilder(pinned=False)
    bb.add_bam_stream(data)
    b = bb.finish(pack=True)
    res = int(b.meta_planes), len(np.unique(bb.lengths()))
    bb.close()
    return res


def test_inputs_are_reproducible():
    for name, (f, seed) in INPUTS.items():
        assert hashlib.sha256(f(seed).tobytes()).hexdigest() == hashlib.sha256(dataset(name)[0].tobytes()).hexdigest(), name


def test_inputs_reach_every_rewrite_path():
    """staged and fallback blocks, a staged block at the quality staging limit, staged general-path reads longer than RW_GORIG,
    missing (0xff) and above -U qualities in staged single-M reads, per-record planes built with many length codes and not built"""
    p = {name: rewrite_paths(dataset(name)[2]) for name in INPUTS}
    assert p["mixed"]["staged"] > 10 and p["boundary"]["staged"] > 10, p
    assert p["mixed"]["fallback"] > 10 and p["long"]["fallback"] > 10 and p["boundary"]["fallback"] > 0, p
    assert p["boundary"]["max_staged_qbytes"] > RW_QCAP - 32, p                 # whole blocks of 161-168-base reads
    assert p["boundary"]["min_fallback_qbytes"] <= RW_QCAP + 16 + 400, p        # one read over
    assert p["boundary"]["staged_general_long"] > 20 and p["mixed"]["staged_general_long"] > 20, p
    assert p["boundary"]["staged_simple_ff"] > 5 and p["boundary"]["staged_simple_above_U"] > 0 and p["mixed"]["staged_simple_above_U"] > 0, p
    lg = p["long"]
    assert lg["max_len"] > 65535 and lg["max_ops"] > 254 and lg["distinct_lengths"] > 256, lg
    planes = {name: meta_planes(dataset(name)[0]) for name in INPUTS}
    assert planes["mixed"][0] == 1 and planes["mixed"][1] == len(MIXED_LENGTHS), planes
    assert planes["boundary"][0] == 1 and planes["boundary"][1] > 1, planes
    assert planes["long"][0] == 0, planes


# ---- the emulated pipeline against the pinned oracle ------------------------------------------------------------------------------------
ARGS = [["-9"], ["-1"], ["-1", "-B"], ["-3", "-U35", "-Y0.2"], ["-5", "-q30"], ["-3", "-P1.5"], ["-7", "-p8"], ["-9", "-p0"]]
CUTS = [None, "211", "gpus3"]


@pytest.mark.parametrize("args", ARGS, ids=lambda a: "".join(a))
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_emulated_pipeline_against_oracle(name, args):
    """uncut, cut every 211 records (every call replays a halo of the reads still open, up to 80 kb long), and spread over three
    emulated devices"""
    data, bb, batch, m = dataset(name)
    ref = oracle(data, args)
    for cut in CUTS:
        env = {"EMU_DEVICES": "8", "CRUMBLE_GPUS": "3"} if cut == "gpus3" else {"CRUMBLE_BATCH_READS": cut} if cut else {}
        r = run_oracle(data, args, binary=EMU_BIN, kind="emu", env_extra=env)
        nbad = int((r["qual"][m] != ref["qual"][m]).sum())
        assert nbad == 0, f"{cut}: {nbad} quality bytes differ"
        assert r["bed"] == ref["bed"], cut
        assert r["counters"] == ref["counters"], cut
