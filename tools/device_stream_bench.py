"""Streams of device records (cg_stream_device) against one call on the whole batch (cg_process_device), on whole synthetic workloads.

For each workload (C2: chr20 at 30x with -9 and with -1 -B; C4: 1000x amplicon panel, -9), starting from torch tensors on the GPU:
  whole      Crumble.process_device on the whole batch (host clock around the call ending in a synchronise, and CUDA events);
  stream K   a DeviceStream fed K records per push (64 Ki, 256 Ki, 1 Mi, 4 Mi) and closed: the wall time and CUDA-event time of every
             push, the held records and quality bytes after it, and the totals;
  kernels    one more pass per K under torch.profiler (CUDA activity): the summed time of k_stream_plan and k_retain and the bytes they
             move, over NVIDIA's data-sheet HBM3e figure for one B200 (7.7 TB/s: a bound, not a measurement).
The sha256 of all emitted qualities must equal the whole-batch run's.  The card's name, power limit and top SM clock are read (nvidia-smi,
a read-only query) in the same run.  Usage: python tools/device_stream_bench.py [--workloads C2-9,C2-1B,C4-9] [--chunks 65536,...]
[--repeats 3] [--out FILE]"""
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
WORKLOADS = {"C2-9": ("C2", ["-9"]), "C2-1B": ("C2", ["-1", "-B"]), "C4-9": ("C4", ["-9"])}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], stdout=subprocess.PIPE,
                           stderr=subprocess.PIPE, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else f"nvidia-smi failed: {r.stderr.strip()}"
    except (OSError, subprocess.TimeoutExpired) as e:
        return f"nvidia-smi failed: {e}"


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "n": len(xs)} if xs else None


def stream_pass(g, chunks, torch, timed):
    """one whole stream; per push: wall ms, event ms, emitted records, held records and bytes"""
    st = g.device_stream()
    q, pushes = [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_all = time.perf_counter()
    for ch in chunks + [None]:
        torch.cuda.synchronize()
        t0 = time.perf_counter(); e0.record()
        r = st.push(ch) if ch is not None else st.close()
        e1.record(); torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        q.append(r["qual"])
        if timed:
            pushes.append({"wall_ms": round(wall, 3), "event_ms": round(e0.elapsed_time(e1), 3), "n_records": r["n_records"],
                           "held_records": r["held_records"], "held_qual_bytes": st.held_qual_len})
    total = (time.perf_counter() - t_all) * 1e3
    sha = hashlib.sha256(torch.cat(q).cpu().numpy().tobytes()).hexdigest()
    return sha, total, pushes


def kernel_times(g, chunks, torch):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sha, _, pushes = stream_pass(g, chunks, torch, True)
    out = {}
    for e in prof.key_averages():
        for k in ("k_stream_plan", "k_retain", "k_stream_keep", "k_ingest", "k_emit"):
            if e.key.startswith(k + "("):
                t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
                out[k] = {"ms": round(t / 1e3, 4), "calls": e.count}
    return out, pushes


def run(name, chunk_sizes, repeats):
    import torch
    import crumble_b200 as cb
    from test_device_batch import params_from_opts
    preset, args = WORKLOADS[name]
    data, n_reads, n_bases = cb.simulate(preset, 1.0, seed=100)
    bb = cb.BatchBuilder(pinned=True); bb.add_bam_stream(data); batch = bb.finish()
    del data
    g = cb.Crumble(params_from_opts(args, ["chr20"]), device=0)
    t = cb.device_batch(batch, 0)
    n = int(batch.n_reads)
    bb.close()
    out = torch.empty_like(t["qual"])
    g.process_device(t, out=out)                                # warm-up
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    wall, ev = [], []
    for _ in range(repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); e0.record()
        g.process_device(t, out=out)
        e1.record(); torch.cuda.synchronize()
        wall.append((time.perf_counter() - t0) * 1e3); ev.append(e0.elapsed_time(e1))
    whole_sha = hashlib.sha256(out.cpu().numpy().tobytes()).hexdigest()
    res = {"workload": name, "args": " ".join(args), "records": n, "quality_bytes": int(t["qual"].numel()),
           "whole": {"wall_ms": stats(wall), "event_ms": stats(ev), "sha256": whole_sha}, "streams": []}
    for k in chunk_sizes:
        chunks = cb.split_device_batch(t, k)
        stream_pass(g, chunks, torch, False)                    # warm-up: buffers grown to their size for this K
        totals, shas, pushes = [], set(), None
        for _ in range(repeats):
            sha, total, pushes = stream_pass(g, chunks, torch, True)
            totals.append(total); shas.add(sha)
        kern, kp = kernel_times(g, chunks, torch)
        held_rec = sum(p["held_records"] for p in kp)
        held_q = sum(p["held_qual_bytes"] for p in kp)
        # k_retain reads and writes every held record: its quality and sequence bytes and 17 bytes of per-record fields (the padding to 8
        # bytes and the CIGARs are left out, so this is a lower bound); k_stream_plan reads tid, pos and rspan of every working record
        retain_bytes = 2 * (held_q + (held_q + 1) // 2 + 17 * held_rec)
        plan_bytes = 12 * (n + held_rec)
        for kk, b in (("k_retain", retain_bytes), ("k_stream_plan", plan_bytes)):
            if kk in kern and kern[kk]["ms"] > 0:
                kern[kk]["bytes"] = b
                kern[kk]["TB_per_s"] = round(b / (kern[kk]["ms"] * 1e-3) / 1e12, 4)
                kern[kk]["share_of_7.7TBs"] = round(b / (kern[kk]["ms"] * 1e-3) / 1e12 / HBM_TBS, 5)
        ok = shas == {whole_sha}
        res["streams"].append({"records_per_push": k, "pushes": len(chunks) + 1, "sha256_equal_to_whole": ok,
                               "total_wall_ms": stats(totals), "max_held_records": max(p["held_records"] for p in pushes),
                               "per_push_last_repeat": pushes, "kernels_profiled_pass": kern})
        print(f"{name} K={k}: {len(chunks) + 1} pushes, total {stats(totals)['median']:.1f} ms (whole {stats(wall)['median']:.1f} ms), "
              f"max held {res['streams'][-1]['max_held_records']}, sha ok {ok}", flush=True)
        if not ok:
            raise SystemExit(f"{name} K={k}: the stream's qualities differ from the whole-batch run")
    g.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="C2-9,C2-1B,C4-9")
    ap.add_argument("--chunks", default="65536,262144,1048576,4194304")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this measurement needs the GPU")
    doc = {"card": card(), "torch": torch.__version__, "hbm_datasheet_TBs": HBM_TBS,
           "workloads": [run(w, [int(x) for x in a.chunks.split(",")], a.repeats) for w in a.workloads.split(",")]}
    doc["card_after"] = card()
    s = json.dumps(doc, indent=1)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(s + "\n")
    print(s if not a.out else f"wrote {a.out}")


if __name__ == "__main__":
    main()
