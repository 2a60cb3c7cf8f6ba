"""Records already in GPU memory (cg_process_device) against the two host-memory paths, on whole synthetic workloads.

For each workload (C2: chr20 at 30x, -9; C4: 1000x amplicon panel, -9) it times, after warm-up and over several repeats:
  resident   cg_run on a batch cg_upload left on the device (the kernel chain alone),
  host e2e   cg_process from pinned host arrays into a pinned host buffer,
  device     Crumble.process_device from torch tensors into a torch tensor (ingest + chain + emit),
and reports the ingest and emit kernels (cg_last_ms CG_T_H2D / CG_T_D2H after a device call) with the bytes they move over their time,
next to NVIDIA's data-sheet HBM3e figure for one B200 (7.7 TB/s: a bound, not a measurement).  It checks that the device path's qualities
have the same sha256 as cg_process's.  The card's name, power limit and top SM clock are read (nvidia-smi, a read-only query) in the
same run.  Usage: python tools/device_batch_bench.py [--workloads C2,C4] [--repeats 5] [--warmup 2] [--out FILE]"""
import argparse
import hashlib
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

HBM_TBS = 7.7
WORKLOADS = {"C2": ("C2", 1.0, 9), "C3": ("C3", 1.0, 1), "C4": ("C4", 1.0, 9)}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi failed: {e}"


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "n": len(xs)}


def run(name, repeats, warmup):
    import numpy as np
    import torch
    import crumble_b200 as cb
    from test_device_batch import params_from_opts
    from test_gpu_device_batch import strip
    preset, scale, level = WORKLOADS[name]
    args = [f"-{level}"] + (["-B"] if name == "C3" else [])
    data, n_reads, n_bases = cb.simulate(preset, scale, seed=100)
    bb = cb.BatchBuilder(pinned=True); bb.add_bam_stream(data); batch = bb.finish()
    del data
    g = cb.Crumble(params_from_opts(args, ["chr20"]), device=0)
    qout = torch.empty(max(int(batch.qual_bytes), 1), dtype=torch.uint8, pin_memory=True).numpy()

    # resident chain
    g.upload(batch)
    for _ in range(warmup):
        g.run()
    resident, chain_dev = [], []
    for _ in range(repeats):
        t0 = time.perf_counter(); g.run(); resident.append((time.perf_counter() - t0) * 1e3); chain_dev.append(g.ms("total"))

    # host memory end to end
    for _ in range(warmup):
        ref = g.process(batch, pinned_out=qout)
    host = []
    for _ in range(repeats):
        t0 = time.perf_counter(); ref = g.process(batch, pinned_out=qout); host.append((time.perf_counter() - t0) * 1e3)
    ref_sha = hashlib.sha256(strip(batch, ref["qual"]).tobytes()).hexdigest()

    # device memory end to end
    t = cb.device_batch(batch, 0)
    out = torch.empty_like(t["qual"])
    torch.cuda.synchronize()
    for _ in range(warmup):
        r = g.process_device(t, out=out)
    dev, dev_ev, ingest, emit, chain2 = [], [], [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); e0.record()
        r = g.process_device(t, out=out)
        e1.record(); torch.cuda.synchronize()
        dev.append((time.perf_counter() - t0) * 1e3); dev_ev.append(e0.elapsed_time(e1))
        ingest.append(g.ms("h2d")); emit.append(g.ms("d2h")); chain2.append(g.ms("total"))
    assert g.h2d_bytes() == 0
    dev_sha = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
    same = dev_sha == ref_sha and np.array_equal(r["events"], ref["events"]) and r["counters"] == ref["counters"]

    n = int(batch.n_reads)
    qual_len, seq_len, padded = int(t["qual"].numel()), int(t["seq"].numel()), int(batch.qual_bytes)
    # ingest: the caller's qualities and sequences in, the padded working arrays out, l_qseq + off + two source offsets per record
    ingest_bytes = qual_len + seq_len + padded + padded // 2 + 28 * n
    # emit: the rewritten qualities in (working layout, only the record's bytes), the caller's array out, l_qseq + off + offset per record
    emit_bytes = 2 * qual_len + 20 * n
    mi, me = stats(ingest)["median"], stats(emit)["median"]
    g.close(); bb.close()
    return {
        "workload": name, "options": " ".join(args), "records": n, "aligned_bases": n_bases, "qual_len": qual_len, "seq_len": seq_len,
        "padded_qual_bytes": padded,
        "resident_cg_run_ms": stats(resident), "resident_chain_device_ms": stats(chain_dev),
        "cg_process_host_e2e_ms": stats(host),
        "process_device_e2e_ms": stats(dev), "process_device_e2e_cuda_event_ms": stats(dev_ev), "process_device_chain_ms": stats(chain2),
        "ingest_ms": stats(ingest), "emit_ms": stats(emit),
        "ingest_bytes": ingest_bytes, "emit_bytes": emit_bytes,
        "ingest_TBps": ingest_bytes / (mi * 1e-3) / 1e12 if mi > 0 else None,
        "emit_TBps": emit_bytes / (me * 1e-3) / 1e12 if me > 0 else None,
        "ingest_share_of_datasheet_hbm": ingest_bytes / (mi * 1e-3) / (HBM_TBS * 1e12) if mi > 0 else None,
        "emit_share_of_datasheet_hbm": emit_bytes / (me * 1e-3) / (HBM_TBS * 1e12) if me > 0 else None,
        "qual_sha256_process_device": dev_sha, "qual_sha256_cg_process": ref_sha, "same_results_as_cg_process": bool(same),
    }


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--workloads", default="C2,C4")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON here")
    a = ap.parse_args()
    res = {"measured_on": card(), "query": "nvidia-smi --query-gpu=name,power.limit,clocks.max.sm",
           "hbm_datasheet_TBps": HBM_TBS, "hbm_note": "7.7 TB/s is NVIDIA's data-sheet HBM3e figure for one B200, a bound, not a measured rate",
           "timing": "host clock around calls that end in a device synchronise; CUDA events for the device call and for the ingest / emit kernels",
           "repeats": a.repeats, "warmup": a.warmup,
           "runs": [run(w, a.repeats, a.warmup) for w in a.workloads.split(",")]}
    res["measured_on_after"] = card()
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(txt + "\n")
    if not all(r["same_results_as_cg_process"] for r in res["runs"]):
        sys.exit("process_device results differ from cg_process")


if __name__ == "__main__":
    main()
