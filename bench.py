#!/usr/bin/env python
"""bench.py — aligned bases/s through the consensus + quality-rewrite hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload C2] [--scale S]

One "step" = one pass of the whole kernel chain (cg_run) over one resident batch of
synthetic aligned reads (default: BASELINE.json configs[1] = crumble -9 on a 64 Mb,
30x chr20-like contig, 2x150 bp; ~1.28e7 reads, ~1.9e9 aligned bases).  N>1: one process
per GPU (torchrun), STRONG scaling: rank r owns region shard r of the one contig with its read
halo; the state-free part of the chain runs on all GPUs at once, the 128-byte state goes from
rank to rank through host shared memory, the rest runs at once again (no device collective;
torch.distributed only for the barrier and the max/sum of the results).

Keys beyond the base contract: roofline (dominant kernel vs measured HBM peak),
cpu_baseline (the reference's own code, oracle/_ref, on this box's host cores),
e2e (host buffers in -> host buffers out through the C ABI), clocks, gpu_launches.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

WORKLOADS = {
    # name: (preset, level args, description)
    "C1": ("C1", ["-9"], "crumble -9, synthetic 1 Mb region, 30x 2x150bp"),
    "C2": ("C2", ["-9"], "crumble -9, synthetic chr20 (64 Mb) 30x 2x150bp"),
    "C3": ("C3", ["-1", "-B"], "crumble -1 -B, synthetic chr20 (64 Mb) 30x"),
    "C4": ("C4", ["-9"], "crumble -9, 1000x amplicon panel (200 x 250 bp)"),
    # run as ONE process driving all GPUs through the C scheduler (cgm_process): python bench.py --workload C5 --gpus 8 [--scale 0.0625]
    "C5": ("C5", ["-9"], "crumble -9, synthetic whole genome 30x: 24 contigs with human chromosome length ratios"),
}


def level_params(cb, args):
    import ctypes as C
    p = cb.default_params()
    for a in args:
        if a[1] in "135789":
            cb.load_lib().cg_params_level(C.byref(p), int(a[1]))
        elif a == "-B":
            p.binary_qual = 1
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile(prefix="clocks", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 7:
                    continue
                try:
                    sm.append(float(f[0])); mx.append(float(f[1]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = float(np.median(sm)); out["sm_max_mhz"] = float(max(mx)); out["reasons"] = sorted(reasons)
            out["samples"] = len(sm)
        return out


def bind_near_gpu(local):
    """Run this rank (and allocate its pinned buffers) on the CPUs of the NUMA node its GPU hangs off: with one rank per GPU the
    host side of every copy then stays on the local socket.  Best effort: any missing piece of sysfs leaves the affinity alone."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local).pci_bus_id if hasattr(torch.cuda.get_device_properties(local), "pci_bus_id") else None
        dom = getattr(torch.cuda.get_device_properties(local), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local), "pci_device_id", 0)
        if bus is None:
            return None
        path = Path(f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0")
        node = int((path / "numa_node").read_text().strip())
        if node < 0:
            return None
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception:  # noqa: BLE001
        return None


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(kernel, workload, scale):
    """DRAM bytes of one launch of the dominant kernel from the committed ncu capture (None when not captured at this size)."""
    try:
        return json.load(open(ROOT / "profiles" / "traffic.json"))[kernel].get(f"{workload}@{scale}")
    except Exception:
        return None


def ref_binary():
    p = ROOT / "oracle" / "_ref" / "crumble_ref"
    if p.exists():
        return p, "reference"
    p = ROOT / "oracle" / "bin" / "crumble_oracle"
    if p.exists():
        return p, "port"
    return None, None


def run_ref_once(binary, path, args):
    env = dict(os.environ); env["CRUMBLE_REF_TIMING"] = "1"
    r = subprocess.run([str(binary), "-z"] + args + ["-O", "bam,raw", path, "mem:discard"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True, env=env)
    if r.returncode != 0:
        raise RuntimeError("reference run failed: " + r.stderr[-500:])
    for line in r.stderr.splitlines():
        if line.startswith("transcode_seconds="):
            return float(line.split("=")[1])
    return None


def cpu_baseline(cb, workload, sample_mb=12.0):
    """Reference transcode() (oracle/_ref, single thread as the reference is) on a bounded sample."""
    binary, kind = ref_binary()
    if binary is None:
        return None
    preset, args, _ = WORKLOADS[workload]
    scale = sample_mb / 64.0 if preset in ("C2", "C3") else (sample_mb if preset == "C1" else (sample_mb / 3096.0 if preset == "C5" else 0.5))
    data, nr, nb = cb.simulate(preset, scale, seed=4242)
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        path = os.path.join(td, "sample.ubam")
        data.tofile(path)
        secs = run_ref_once(binary, path, args)
    return {"value": nb / secs, "unit": "aligned bases/s", "cores": 1, "kind": kind,
            "sample": f"{preset} x{scale:.4g} seed 4242: {nr} reads, {nb} aligned bases, transcode() {secs:.2f} s (memory-backed reader, discarding writer)"}


def parity_gate(cb, g, workload):
    """Part of the cpu_baseline leg: a small sample of the workload through the reference (oracle/_ref) AND through the context the bench
    has just timed; every quality byte, the BED text and the 19 counters must be equal.  Never raises: the outcome is a string in the
    bench line (the full-size comparison lives in tests/test_gpu_full_size.py)."""
    try:
        sys.path.insert(0, str(ROOT / "tests"))
        from util import run_oracle, valid_mask
        preset, args, _ = WORKLOADS[workload]
        scale = {"C1": 0.5, "C2": 1 / 128, "C3": 1 / 128, "C4": 0.05}.get(preset, 1 / 128)
        data, nr, nb = cb.simulate(preset, scale, seed=777)
        bb = cb.BatchBuilder(pinned=False); bb.add_bam_stream(data)
        batch = bb.finish(pack=True)
        out = g.process(batch)
        ref = run_oracle(data, args)
        m = valid_mask(bb)
        nbad = int((out["qual"][m] != ref["qual"][m]).sum())
        ok = nbad == 0 and cb.bed_text(out["events"], ref["names"]) == ref["bed"] and out["counters"] == ref["counters"]
        bb.close()
        return (("bit-exact" if ok else f"MISMATCH ({nbad} quality bytes differ)") +
                f" vs oracle ({ref['kind']}) on {preset} x{scale:.4g} seed 777: {nr} reads, every quality byte, BED text, 19 counters")
    except Exception as e:  # noqa: BLE001
        return f"not checked here ({type(e).__name__}: {e}); see tests/test_gpu_full_size.py"


def reference_shards(preset, scale, nproc):
    """The workload cut into nproc independent pieces of equal size for the all-cores reference arm (how users parallelise crumble:
    one process per region).  The pieces together are the SAME amount and kind of data the GPU arm processes in one step."""
    if preset == "C4":                                             # amplicons are independent: split their number
        n_amp = max(1, int(200 * scale))
        nproc = min(nproc, n_amp)
        return [("C4", (n_amp // nproc + (1 if i < n_amp % nproc else 0)) / 200.0) for i in range(nproc)]
    return [(preset, scale / nproc)] * nproc


def bench_reference(a, rank, world):
    """--impl reference: the reference's own CPU implementation (oracle/_ref: snp_score.c compiled from the reference's sources) on all
    host cores, one single-threaded process per piece, on the same workload size as the GPU arm.  The step time is the slowest
    piece's transcode() (memory-backed reader, discarding writer: what cpu_baseline times too), all pieces running at once."""
    if rank != 0:
        return
    import crumble_b200 as cb
    binary, kind = ref_binary()
    if binary is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle binaries not built"}))
        return
    preset, args, desc = WORKLOADS[a.workload]
    cores = os.cpu_count() or 1
    nproc = max(1, min(cores, 64))
    pieces = reference_shards(preset, a.scale, nproc)
    tmpdir = "/dev/shm" if os.path.isdir("/dev/shm") else None
    with tempfile.TemporaryDirectory(dir=tmpdir) as td:
        paths, bases = [], 0
        for i, (pr, sc) in enumerate(pieces):
            data, nr, nb = cb.simulate(pr, sc, seed=9000 + i)
            p = os.path.join(td, f"s{i}.ubam"); data.tofile(p); paths.append(p); bases += nb
            del data

        def step():
            t0 = time.perf_counter()
            env = dict(os.environ); env["CRUMBLE_REF_TIMING"] = "1"
            procs = [subprocess.Popen([str(binary), "-z"] + args + ["-O", "bam,raw", p, "mem:discard"],
                                      stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True, env=env) for p in paths]
            secs = []
            for pr in procs:
                err = pr.communicate()[1]
                if pr.returncode != 0:
                    raise RuntimeError("reference piece failed: " + err[-300:])
                m = [l for l in err.splitlines() if l.startswith("transcode_seconds=")]
                secs.append(float(m[0].split("=")[1]) if m else None)
            wall = time.perf_counter() - t0
            return (max(secs) if all(x is not None for x in secs) else wall), wall
        for _ in range(a.warmup):
            step()
        ts = [step() for _ in range(a.steps)]
    tot = sum(t[0] for t in ts); wall = sum(t[1] for t in ts)
    v = bases * a.steps / tot
    line = {"impl": "reference", "metric": "aligned bases/sec (consensus+qual rewrite)", "value": v, "unit": "aligned bases/s",
            "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True,
            "scaling": "strong" if a.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64+u8", "data": "synthetic",
            "config": {"workload": desc + (f" (scale {a.scale})" if a.scale != 1.0 else ""),
                       "pieces": f"{len(pieces)} x {preset} x{pieces[0][1]:.4g} ({bases} aligned bases per step = the whole workload), one single-threaded reference process per piece, all at once",
                       "wall_ms_per_step": 1e3 * wall / a.steps},
            "cpu_baseline": {"value": v, "unit": "aligned bases/s", "cores": len(pieces), "kind": kind,
                             "sample": f"the whole workload: {len(pieces)} concurrent reference processes, step = slowest piece's transcode() (memory-backed reader, discarding writer)"},
            "e2e": {"value": v, "unit": "aligned bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


class Mailbox:
    """128-byte messages between the ranks of one box through a shared-memory file: the carry of a region shard travels to the rank on
    its right.  No device collective is involved (SURVEY.md 8e): NCCL is used for the barrier and the reductions of the results only.
    Every sender owns a ring of RING slots (message of step s in slot s % RING) and every receiver publishes the last step it has
    consumed: a sender never overwrites a message its neighbour has not read yet, however far the ranks drift apart (rank 0 waits
    for nobody's carry, so without this it can run whole steps ahead)."""

    RING = 8
    MSG = 8 + 128
    SLOT = 8 + RING * MSG                                        # [consumed step of this rank as a receiver][RING x (step, payload)]

    def __init__(self, world, rank, key):
        self.path = f"/dev/shm/crumble_mbox_{key}"
        self.world, self.rank = world, rank
        if rank == 0:
            np.zeros(world * self.SLOT, np.uint8).tofile(self.path)

    def open(self):
        self.m = np.memmap(self.path, dtype=np.uint8, mode="r+", shape=(self.world * self.SLOT,))

    def _i64(self, byte_off):
        return self.m[byte_off: byte_off + 8].view(np.int64)

    def _wait(self, ready, what, timeout_s=300.0):
        """spin (the carry is on the critical path of every step); a neighbour that died must not hang the job"""
        n = 0
        t0 = None
        while not ready():
            n += 1
            if n & 0xfff == 0:
                if t0 is None:
                    t0 = time.perf_counter()
                elif time.perf_counter() - t0 > timeout_s:
                    raise RuntimeError(f"mailbox: rank {self.rank} waited more than {timeout_s:.0f} s for {what}")

    def send(self, step, blob):
        """to rank + 1; steps count from 1"""
        ack = self._i64((self.rank + 1) * self.SLOT)
        self._wait(lambda: int(ack[0]) >= step - self.RING, f"rank {self.rank + 1} to consume step {step - self.RING}")   # the slot still holds an unread message
        o = self.rank * self.SLOT + 8 + (step % self.RING) * self.MSG
        self.m[o + 8: o + self.MSG] = np.frombuffer(blob, np.uint8)
        self._i64(o)[0] = step                                   # x86: stores stay in program order

    def recv(self, step, src):
        o = src * self.SLOT + 8 + (step % self.RING) * self.MSG
        q = self._i64(o)
        self._wait(lambda: int(q[0]) == step, f"the carry of step {step} from rank {src}")
        blob = self.m[o + 8: o + self.MSG].tobytes()
        self._i64(self.rank * self.SLOT)[0] = step               # consumed
        return blob

    def close(self):
        if self.rank == 0:
            try:
                os.unlink(self.path)
            except OSError:
                pass


def rank_shard(cb, preset, scale, seed, rank, world, threads, pack):
    """This rank's region shard of the workload's single contig, generated on its own (the generator makes the reads of each 256 kb chunk from
    the chunk's own random stream, and the chunks concatenate to exactly the full stream): the reads starting in its chunks, the read halo
    out of the chunk before, and the column window.  Cuts: X = first read of the right neighbour, S = start of the first read of this
    shard that reaches X (include/crumble_gpu.h)."""
    import ctypes as C
    CH = 1 << 18
    cfg = cb.api.SimCfg(); cb.api.load_sim().simgen_preset(C.byref(cfg), preset.encode(), scale, seed)
    assert cfg.n_contigs == 1 and not cfg.amplicon, "region shards over the ranks need a single-contig workload"
    njobs = (int(cfg.contig_len) + CH - 1) // CH
    a, b = njobs * rank // world, njobs * (rank + 1) // world
    jf, jl = max(a - 1, 0), min(b + 1, njobs)
    data, _, _ = cb.simulate(preset, scale, seed, threads=threads, job_first=jf, job_count=jl - jf)
    bb = cb.BatchBuilder(pinned=True); bb.add_bam_stream(data); del data
    batch = bb.finish(pack=pack)
    n = int(batch.n_reads)
    pos = np.ctypeslib.as_array(batch.pos, shape=(n,)); tid = np.ctypeslib.as_array(batch.tid, shape=(n,))
    npl = int(np.searchsorted(-tid, 1))                          # placed records come first (tid 0), the unmapped tail (-1) last
    end = cb.batch_ends(batch)
    r0 = int(np.searchsorted(pos[:npl], a * CH)) if rank > 0 else 0
    r1 = int(np.searchsorted(pos[:npl], b * CH)) if rank < world - 1 else n
    sh = {"r0": r0, "r1": r1, "h0": r0, "first": 1, "lo_tid": -1, "lo_pos": 0, "cnt_pos": 0, "hi_tid": -1, "hi_pos": 0, "next_lo_pos": 0}
    if rank > 0:
        X = int(pos[r0]); reach = np.nonzero(end[:r0] > X)[0]
        S = int(pos[reach[0]]) if reach.size else X
        h = np.nonzero(end[:r0] > S)[0]
        sh.update(first=0, lo_tid=0, lo_pos=S, cnt_pos=X, h0=int(h[0]) if h.size else r0)
    if rank < world - 1:
        X = int(pos[r1]); reach = np.nonzero(end[sh["h0"]:r1] > X)[0]
        S = int(pos[sh["h0"] + reach[0]]) if reach.size else X
        sh.update(hi_tid=0, hi_pos=X, next_lo_pos=S)
    sub, keep = cb.sub_batch(batch, sh["h0"], r1)
    lq = np.ctypeslib.as_array(batch.l_qseq, shape=(n,))
    inp = end > pos
    own = np.zeros(n, bool); own[r0:r1] = True
    nc = np.ctypeslib.as_array(batch.n_cigar, shape=(n,)).astype(np.int64)
    bases = int(lq[own & inp].sum())
    algo = int((((lq + 1) >> 1) + 2 * lq.astype(np.int64) + 4 * nc + 16)[own & inp].sum())
    # the records this rank finalises, in order: halo records still open at its left cut and closed here, own records closed here
    openL = np.zeros(n, bool)
    if rank > 0:
        openL[:r0] = inp[:r0] & (end[:r0] > sh["cnt_pos"])
    openR = inp & (end > sh["hi_pos"]) if rank < world - 1 else np.zeros(n, bool)
    final = (own | openL) & ~openR
    final[: sh["h0"]] = False
    return dict(bb=bb, batch=batch, sub=sub, keep=keep, sh=sh, bases=bases, algo=algo, final=np.nonzero(final)[0], reads=int(own.sum()),
                chunks=(a, b), CH=CH, njobs=njobs)


def bench_shards(a, rank, world, local):
    """N > 1: STRONG scaling of the workload's one contig.  Rank r owns region shard r (cg_shard_begin / _carry / _end, include/crumble_gpu.h):
    the state-free 3/4 of the chain runs on all GPUs at once, the 128-byte state goes from rank to rank, the rest runs at once again.
    value = total aligned bases / slowest rank, batch resident in HBM; e2e = the same from pinned host buffers to pinned host buffers."""
    import hashlib
    import torch
    import torch.distributed as dist
    import crumble_b200 as cb
    torch.cuda.set_device(local)
    numa = bind_near_gpu(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    preset, args, desc = WORKLOADS[a.workload]
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    t_gen = time.perf_counter()
    R = rank_shard(cb, preset, a.scale, 100, rank, world, max(1, (os.cpu_count() or 1) // world), not a.no_pack)
    t_gen = time.perf_counter() - t_gen
    sub, sh = R["sub"], R["sh"]
    win = cb.shard_window(sh)
    g = cb.Crumble(level_params(cb, args), device=local)
    stream = torch.cuda.Stream(device=local)
    g.set_stream(stream.cuda_stream)
    mbox = Mailbox(world, rank, os.environ.get("MASTER_PORT", "0"))
    qout = torch.empty(max(int(sub.qual_bytes), 1), dtype=torch.uint8, pin_memory=True).numpy()

    def barrier():
        torch.cuda.synchronize(); dist.barrier(); torch.cuda.synchronize()

    barrier(); mbox.open(); barrier()
    seq = [0]

    phase_s = [0.0, 0.0, 0.0, 0.0]                               # host wall clock per phase (CG_BENCH_PHASES=1 prints them): begin, wait, carry, end

    def step(resident):
        seq[0] += 1
        t0 = time.perf_counter()
        g.shard_begin(None if resident else sub, win, pinned_out=None if resident else qout)
        t1 = time.perf_counter()
        cin = mbox.recv(seq[0], rank - 1) if rank > 0 else None
        t2 = time.perf_counter()
        cout = g.shard_carry(cin, want_out=rank < world - 1)
        if rank < world - 1:
            mbox.send(seq[0], cout)
        t3 = time.perf_counter()
        r = g.shard_end()
        t4 = time.perf_counter()
        for i, d in enumerate((t1 - t0, t2 - t1, t3 - t2, t4 - t3)):
            phase_s[i] += d
        return r

    def timed(resident, steps, warmup):
        for _ in range(warmup):
            step(resident)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        ev0.record(stream)
        tm = {}
        for _ in range(steps):
            out = step(resident)
            if resident:
                for k, v in g.timers().items():
                    tm[k] = tm.get(k, 0.0) + v / steps
        ev1.record(stream)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if resident:                                             # device clock on the launching stream (idle gaps waiting for the left neighbour included)
            dt = ev0.elapsed_time(ev1) * 1e-3
        barrier()
        t = torch.tensor([dt], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), out, tm

    g.upload(sub)
    sampler = ClockSampler(local); sampler.start()
    dev_s, out_r, stage = timed(True, a.steps, a.warmup)
    clocks = sampler.stop()
    if os.environ.get("CG_BENCH_PHASES"):
        n_st = a.steps + a.warmup
        sys.stderr.write(f"[phases] rank {rank}: begin {phase_s[0] / n_st * 1e3:.3f} wait {phase_s[1] / n_st * 1e3:.3f} carry {phase_s[2] / n_st * 1e3:.3f} "
                         f"end {phase_s[3] / n_st * 1e3:.3f} ms per step; stages {({k: round(v, 3) for k, v in stage.items()})}\n")
    launches = g.launches() * a.steps
    e2e_s, out, _ = timed(False, a.e2e_steps, 1)
    h2d = g.h2d_bytes()
    # ---- totals over the ranks ----
    vec = torch.tensor([float(R["bases"]), float(R["algo"]), float(stage.get("columns", 0.0)), float(h2d), float(sub.qual_bytes), float(launches), float(R["reads"])],
                       dtype=torch.float64, device="cuda")
    tot = vec.clone(); dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    mx = vec.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    bases, algo = float(tot[0].item()), float(tot[1].item())
    col_ms = float(mx[2].item())
    # ---- parity (outside the timed regions): every rank hashes the qualities of the records it finalises; rank 0 runs the whole contig
    # through one context and hashes the same records ----
    off = np.ctypeslib.as_array(R["batch"].off, shape=(int(R["batch"].n_reads),)); lq = np.ctypeslib.as_array(R["batch"].l_qseq, shape=(int(R["batch"].n_reads),))
    base = int(off[sh["h0"]])
    hsh = hashlib.sha256()
    for i in R["final"]:
        hsh.update(out["qual"][int(off[i]) - base: int(off[i]) - base + int(lq[i])].tobytes())
    mine = (hsh.hexdigest(), int(R["final"].size), out["counters"], len(out["events"]), out_r["counters"])
    got = [None] * world
    dist.all_gather_object(got, mine)
    parity = "skipped (--no-parity)"
    if rank == 0 and not a.no_parity:
        t_par = time.perf_counter()
        data, _, _ = cb.simulate(preset, a.scale, 100)
        fb = cb.BatchBuilder(pinned=False); fb.add_bam_stream(data); del data
        full = fb.finish()
        g2 = cb.Crumble(level_params(cb, args), device=local)
        ref = g2.process(full)
        n = int(full.n_reads)
        pos = np.ctypeslib.as_array(full.pos, shape=(n,)); tid = np.ctypeslib.as_array(full.tid, shape=(n,))
        foff = np.ctypeslib.as_array(full.off, shape=(n,)); flq = np.ctypeslib.as_array(full.l_qseq, shape=(n,))
        end = cb.batch_ends(full); inp = end > pos
        npl = int(np.searchsorted(-tid, 1))
        njobs = R["njobs"]
        ok = True; nfinal = 0
        cnt = {k: 0 for k in ref["counters"]}; nev = 0
        for r in range(world):
            ja, jb = njobs * r // world, njobs * (r + 1) // world
            r0 = int(np.searchsorted(pos[:npl], ja * R["CH"])) if r > 0 else 0
            r1 = int(np.searchsorted(pos[:npl], jb * R["CH"])) if r < world - 1 else n
            own = np.zeros(n, bool); own[r0:r1] = True
            openL = np.zeros(n, bool)
            if r > 0:
                openL[:r0] = inp[:r0] & (end[:r0] > int(pos[r0]))
            openR = inp & (end > int(pos[r1])) if r < world - 1 else np.zeros(n, bool)
            idx = np.nonzero((own | openL) & ~openR)[0]
            hh = hashlib.sha256()
            for i in idx:
                hh.update(ref["qual"][int(foff[i]): int(foff[i]) + int(flq[i])].tobytes())
            ok &= hh.hexdigest() == got[r][0] and idx.size == got[r][1]
            nfinal += idx.size
            for c in cnt:
                cnt[c] += got[r][2][c]
            nev += got[r][3]
            ok &= got[r][2] == got[r][4]                          # resident and end-to-end passes agree
        ok &= nfinal == n and cnt == ref["counters"] and nev == len(ref["events"])
        parity = ("bit-exact" if ok else "MISMATCH") + f" vs one context on the whole contig ({n} records, all quality bytes by sha256 per shard, counters, event count; {time.perf_counter() - t_par:.0f} s)"
        g2.close(); fb.close()
    if rank == 0:
        peak, peak_src = measured_peak()
        achieved = algo / (col_ms * 1e-3) / 1e9 if col_ms > 0 else None
        line = {
            "metric": "aligned bases/sec (consensus+qual rewrite)", "value": bases * a.steps / dev_s, "unit": "aligned bases/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * dev_s / a.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64+u8", "data": "synthetic",
            "config": {"workload": desc + (f" (scale {a.scale})" if a.scale != 1.0 else ""), "reads_total": int(tot[6].item()), "aligned_bases_total": int(bases),
                       "sharding": f"{world} region shards of the one contig, one per GPU, read halo at every cut; state-free part of the chain on all GPUs at once, "
                                   "128-byte state from rank to rank (host shared memory, no device collective), the rest at once again",
                       "halo_records": sh["r0"] - sh["h0"], "l2": "inputs per GPU far exceed the 126 MB L2 only at N <= 4; see profiles/ for the per-kernel view",
                       "stage_ms_rank0": {k: round(v, 4) for k, v in stage.items()}, "datagen_s": round(t_gen, 2), "parity": parity},
            "roofline": {"bound": "hbm", "kernel": "k_column", "achieved": achieved, "peak": peak * world, "unit": "GB/s", "frac": (achieved / (peak * world)) if achieved else None,
                         "traffic": None, "algorithmic_bytes_per_launch": int(algo), "kernel_ms": col_ms, "peak_source": peak_src + f" x {world} GPUs; kernel_ms = slowest rank's k_column",
                         "whole_chain_frac": algo / (dev_s / a.steps) / 1e9 / (peak * world)},
            "e2e": {"value": bases * a.e2e_steps / e2e_s, "unit": "aligned bases/s", "h2d_bytes_per_step": int(tot[3].item()), "d2h_bytes_per_step": int(tot[4].item()),
                    "ms_per_step": 1e3 * e2e_s / a.e2e_steps, "steps": a.e2e_steps, "host_binding": numa,
                    "how": "every rank: pinned host buffers of its shard -> cg_shard_begin / _carry / _end -> pinned host qualities; copies inside the timed region"},
            "gpu_launches": int(tot[5].item()), "clocks": clocks,
        }
        print(json.dumps(line))
    barrier()
    mbox.close()
    dist.destroy_process_group()


def bench_genome(a):
    """--workload C5: the whole-genome configuration through the C scheduler of crumble_b200/csrc/cg_multi.c, ONE process and one host thread
    per GPU: the coordinate-sorted batch of all 24 contigs is cut into a.gpus region shards of equal size (cuts inside a contig get a read
    halo, cuts between contigs separate independent pieces), every device downloads its own byte range, the host gathers events and
    counters.  Host buffers in, host buffers out: this is an end-to-end number; `value` repeats it (there is no resident form of this call).
    The full 3.1 Gb at 30x is 9.3e10 aligned bases (250 GB of host arrays): the default scale 1/16 keeps the contig proportions."""
    import torch
    import crumble_b200 as cb
    preset, args, desc = WORKLOADS["C5"]
    scale = a.scale if a.scale != 1.0 else 0.0625
    t_gen = time.perf_counter()
    data, n_reads, n_bases = cb.simulate(preset, scale, seed=100)
    bb = cb.BatchBuilder(pinned=True); bb.add_bam_stream(data); del data
    batch = bb.finish(pack=not a.no_pack)
    t_gen = time.perf_counter() - t_gen
    bases = cb.aligned_bases(batch); algo = cb.algorithmic_bytes(batch)
    params = level_params(cb, args)
    m = cb.MultiCrumble(params, devices=list(range(a.gpus)))
    qout = torch.empty(max(int(batch.qual_bytes), 1), dtype=torch.uint8, pin_memory=True).numpy()
    for _ in range(max(1, min(a.warmup, 2))):
        out = m.process(batch, pinned_out=qout)
    sampler = ClockSampler(0); sampler.start()
    t0 = time.perf_counter(); dev_ms = 0.0
    for _ in range(a.steps):
        out = m.process(batch, pinned_out=qout)
        dev_ms += m.ms()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    h2d = m.h2d_bytes()
    parity = "skipped (--no-parity)"
    if not a.no_parity:
        g = cb.Crumble(params, device=0)
        ref = g.process(batch)
        mask = np.zeros(int(batch.qual_bytes) + 1, np.int8)
        n = int(batch.n_reads); off = np.ctypeslib.as_array(batch.off, shape=(n,)); lq = np.ctypeslib.as_array(batch.l_qseq, shape=(n,))
        np.add.at(mask, off, 1); np.add.at(mask, off + lq, -1); mask = np.cumsum(mask[:-1]) > 0
        ok = np.array_equal(ref["qual"][mask], out["qual"][mask]) and np.array_equal(ref["events"], out["events"]) and ref["counters"] == out["counters"]
        parity = ("bit-exact" if ok else "MISMATCH") + " vs cg_process of the whole batch on one GPU (every quality byte, events, counters)"
        g.close()
    peak, peak_src = measured_peak()
    v = bases * a.steps / dt
    line = {"metric": "aligned bases/sec (consensus+qual rewrite)", "value": v, "unit": "aligned bases/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * dt / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64+u8", "data": "synthetic",
            "config": {"workload": desc + f" (scale {scale}: {n_reads} reads, {int(bases)} aligned bases)", "sharding": f"cgm_process: {a.gpus} region shards of the 24-contig batch, one host thread + one context per GPU, host gather",
                       "slowest_shard_device_ms": dev_ms / a.steps, "datagen_s": round(t_gen, 2), "parity": parity,
                       "note": "value == e2e: the scheduler call takes host buffers; the resident view of the same kernels is the C2 line"},
            "roofline": {"bound": "hbm", "kernel": "whole call", "achieved": algo * a.steps / dt / 1e9, "peak": peak * a.gpus, "unit": "GB/s", "frac": algo * a.steps / dt / 1e9 / (peak * a.gpus),
                         "traffic": None, "algorithmic_bytes_per_launch": int(algo), "peak_source": peak_src + f" x {a.gpus} GPUs"},
            "e2e": {"value": v, "unit": "aligned bases/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(batch.qual_bytes) + 12 * len(out["events"]) + 8 * 19,
                    "ms_per_step": 1e3 * dt / a.steps, "steps": a.steps},
            "gpu_launches": None, "clocks": clocks}
    print(json.dumps(line))


def world_size():
    return int(os.environ.get("WORLD_SIZE", "1"))


DUMP_RECORDS = 1 << 15
DUMP_QUAL_VALUES = 1 << 23                                       # 32 MiB of float32 qualities
DUMP_LIMIT = 64 << 20


def dump_outputs(d, bb, res):
    """What a caller of the timed path receives (cg_download after the last cg_run), as .npy files in d, DUMP_LIMIT bytes at most
    (about 20 MB at C2): the rewritten quality strings of a fixed sample of up to DUMP_RECORDS records (seed 0; float32,
    concatenated in sample order, at most DUMP_QUAL_VALUES values, with each sampled record's index and length), the BED events
    (tid, pos, tag; float64; a fixed sample of rows, seed 1, in list order when the whole list would not fit) and the 19 counters
    (float64, in COUNTER_NAMES order).  The inputs are seeded, so two builds given the same arguments can be compared file for file."""
    import crumble_b200 as cb
    os.makedirs(d, exist_ok=True)
    off, ln = bb.offsets(), bb.lengths()
    idx = np.sort(np.random.default_rng(0).choice(off.size, min(DUMP_RECORDS, off.size), replace=False))
    idx = idx[np.cumsum(ln[idx].astype(np.int64)) <= DUMP_QUAL_VALUES]
    qual = np.concatenate([res["qual"][int(off[i]): int(off[i]) + int(ln[i])] for i in idx]) if idx.size else np.zeros(0, np.uint8)
    ev = res["events"]
    arrays = {"qual_sample": qual.astype(np.float32), "qual_sample_records": idx.astype(np.float64), "qual_sample_lengths": ln[idx].astype(np.float64),
              "counters": np.array([res["counters"][k] for k in cb.COUNTER_NAMES], dtype=np.float64)}
    rows = (DUMP_LIMIT - 4096 - sum(a.nbytes for a in arrays.values())) // 24          # 4096: room for the five .npy headers
    if len(ev) > rows:
        ev = ev[np.sort(np.random.default_rng(1).choice(len(ev), rows, replace=False))]
    arrays["events"] = np.stack([ev["tid"], ev["pos"], ev["tag"]], axis=1).astype(np.float64) if len(ev) else np.zeros((0, 3))
    assert sum(a.nbytes for a in arrays.values()) <= DUMP_LIMIT - 4096
    for name, arr in arrays.items():
        np.save(os.path.join(d, name + ".npy"), arr)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--workload", default="C2")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pack", action="store_true", help="upload the plain 4-bit / 8-bit arrays instead of the batcher's compact planes")
    ap.add_argument("--replicas", action="store_true", help="N > 1: one private copy of the workload per GPU (weak scaling) instead of region shards of one contig")
    ap.add_argument("--no-parity", action="store_true", help="N > 1: skip the whole-contig comparison rank 0 makes after the timed regions")
    ap.add_argument("--dump-outputs", metavar="DIR", help="one GPU: write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl == "reference" or a.workload == "C5" or world_size() > 1):
        raise SystemExit("--dump-outputs is supported for the one-GPU run of the resident chain only")
    if a.warmup < 3 and a.impl != "reference":
        a.warmup = 3
    rank = int(os.environ.get("RANK", "0")); world = world_size()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        if a.workload == "C5" and a.scale == 1.0:
            a.scale = 0.0625
        bench_reference(a, rank, world)
        return
    if a.workload == "C5":
        if world > 1:
            raise SystemExit("--workload C5 is one process driving all GPUs (python bench.py --workload C5 --gpus N), not a torchrun job")
        bench_genome(a)
        return
    if world > 1 and not a.replicas:
        bench_shards(a, rank, world, local)
        return

    import torch
    import crumble_b200 as cb
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU path")
    torch.cuda.set_device(local)
    numa = bind_near_gpu(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    preset, args, desc = WORKLOADS[a.workload]
    t_gen = time.perf_counter()
    data, n_reads, n_bases = cb.simulate(preset, a.scale, seed=100 + rank)
    bb = cb.BatchBuilder(pinned=True)
    bb.add_bam_stream(data)
    del data
    batch = bb.finish(pack=not a.no_pack)                       # compact planes: 2-bit bases + exceptions, dictionary-coded qualities
    t_gen = time.perf_counter() - t_gen
    algo_bytes = cb.algorithmic_bytes(batch)
    bases = cb.aligned_bases(batch)
    g = cb.Crumble(level_params(cb, args), device=local)
    stream = torch.cuda.Stream(device=local)
    g.set_stream(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- resident: inputs already in HBM; K passes of the whole kernel chain ------------------
    g.upload(batch)
    for _ in range(a.warmup):
        g.run()
    sampler = ClockSampler(local); sampler.start()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    col_ms, rew_ms, stage = [], [], {}
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(a.steps):
            g.run()
            t = g.timers()
            col_ms.append(t["columns"]); rew_ms.append(t["rewrite"])
            for k, v in t.items():
                stage[k] = stage.get(k, 0.0) + v / a.steps
        ev1.record(stream)
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = g.launches() * a.steps
    clocks = sampler.stop()
    tmax = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    tot_bases = torch.tensor([float(bases)], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX); dist.all_reduce(tot_bases, op=dist.ReduceOp.SUM)
    dev_ms_max = float(tmax.item()); all_bases = float(tot_bases.item())
    value = all_bases * a.steps / (dev_ms_max * 1e-3)
    if a.dump_outputs:
        res = g.download(batch)
        if res["n_events"] > len(res["events"]):
            res = g.download(batch, events_cap=res["n_events"])
        dump_outputs(a.dump_outputs, bb, res)

    # ---- end to end: pinned host SoA -> C ABI -> host quality buffer, copies inside the timed region
    qout = torch.empty(max(int(batch.qual_bytes), 1), dtype=torch.uint8, pin_memory=True).numpy()
    g.process(batch, pinned_out=qout)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        out = g.process(batch, pinned_out=qout)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = all_bases * a.e2e_steps / float(te.item())
    h2d = g.h2d_bytes(); d2h = int(batch.qual_bytes) + 12 * len(out["events"]) + 8 * 19
    e2e_timers = g.timers()

    if rank == 0:
        peak, peak_src = measured_peak()
        col = float(np.mean(col_ms))
        achieved = algo_bytes / (col * 1e-3) / 1e9
        line = {
            "metric": "aligned bases/sec (consensus+qual rewrite)", "value": value, "unit": "aligned bases/s",
            "n_gpus": world, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dev_ms_max / a.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64+u8", "data": "synthetic",
            "config": {"workload": desc + (f" (scale {a.scale})" if a.scale != 1.0 else ""), "reads_per_gpu": int(batch.n_reads),
                       "aligned_bases_per_gpu": int(bases), "columns_per_gpu": g.n_columns(), "sharding": "one contig shard per GPU, no collective",
                       "l2": "inputs (>= 2.6 B/base resident) far exceed the 126 MB L2; no flush needed",
                       "stage_ms": {k: round(v, 4) for k, v in stage.items()}, "datagen_s": round(t_gen, 2)},
            "roofline": {"bound": "hbm", "kernel": "k_column", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": measured_traffic("k_column", a.workload, a.scale), "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": col, "peak_source": peak_src,
                         "whole_chain_frac": algo_bytes / (dev_ms_max / a.steps * 1e-3) / 1e9 / peak,
                         "frac_of_nominal_8TBs": achieved / 8000.0},
            "e2e": {"value": e2e_value, "unit": "aligned bases/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": 1e3 * float(te.item()) / a.e2e_steps, "h2d_ms": e2e_timers["h2d"], "d2h_ms": e2e_timers["d2h"],
                    "steps": a.e2e_steps, "host_binding": numa,
                    "upload": ("compact planes built by the batcher: 2-bit bases + exception list" + (f", {batch.qual_bits}-bit dictionary-coded qualities" if batch.qual_bits else ", 8-bit qualities (more than 16 distinct values)")) if batch.seq2 else "4-bit bases, 8-bit qualities",
                    "how": "cg_process: per-record arrays, then base data in ~96 MB chunks on a copy stream; slice i of the chain starts "
                    "when chunk i has landed; qualities return on a second copy stream (h2d_ms / d2h_ms are the spans of the two copy streams and overlap)"},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if world == 1 and not a.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline(cb, a.workload)
            except Exception as e:  # noqa: BLE001
                line["cpu_baseline"] = {"error": str(e)}
            line["config"]["parity"] = parity_gate(cb, g, a.workload)
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
