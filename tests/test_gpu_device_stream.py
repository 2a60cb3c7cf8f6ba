"""Streams of device records (cg_stream_device) on the GPU: a stream pushed in chunks gives, concatenated, what one call on the whole
batch gives (cg_process on the same context, the oracle on tiny, process_device by sha256 on whole C2), with bounded held records; deep
columns cut through; a non-default torch stream; one chunk buffer reused for every push; qual_out aliasing the chunk; events fetched again;
calls that must be refused while a stream is open."""
import hashlib

import numpy as np
import pytest

import crumble_b200 as cb
from test_device_batch import params_from_opts
from test_gpu_device_batch import strip
from test_gpu_parity import LEVELS, dataset
from util import run_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def stream_all(g, chunks, events_cap=1 << 16):
    """push every chunk, then close; the concatenated qualities (host), events, summed counters and held records after each push"""
    s = g.device_stream()
    q, ev, cnt, held, nrec = [], [], None, [], 0
    for ch in chunks + [None]:
        r = s.push(ch, events_cap=events_cap) if ch is not None else s.close(events_cap=events_cap)
        q.append(r["qual"].cpu().numpy()); ev.append(r["events"]); held.append(r["held_records"]); nrec += r["n_records"]
        cnt = r["counters"] if cnt is None else {k: cnt[k] + r["counters"][k] for k in cnt}
    assert held[-1] == 0
    return {"qual": np.concatenate(q), "events": np.concatenate(ev), "counters": cnt, "held": held, "n_records": nrec}


def assert_same(ref, got, what=""):
    nbad = int((ref["qual"] != got["qual"]).sum()) if ref["qual"].size == got["qual"].size else -1
    assert nbad == 0, f"{what}: {nbad} quality bytes differ"
    assert np.array_equal(ref["events"], got["events"]), what
    assert ref["counters"] == got["counters"], what


def check_cuts(batch, args, cuts_list, names=("chr1", "chr2")):
    g = cb.Crumble(params_from_opts(args, names), device=0)
    ref = g.process(batch)
    ref["qual"] = strip(batch, ref["qual"])
    t = cb.device_batch(batch, 0)
    n = int(batch.n_reads)
    for cuts in cuts_list:
        got = stream_all(g, cb.split_device_batch(t, cuts=cuts))
        assert got["n_records"] == n
        assert_same(ref, got, f"{' '.join(args)} cuts {cuts[:4]}...")
    g.close()


def every(n, k):
    return list(range(k, n, k))


@pytest.mark.parametrize("args", LEVELS, ids=lambda a: "".join(a))
def test_tiny_against_oracle(args):
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_opts(args), device=0)
    got = stream_all(g, cb.split_device_batch(cb.device_batch(batch, 0), 997))
    ref = run_oracle(data, args)
    assert int((got["qual"] != ref["qual"][mask]).sum()) == 0, f"quality bytes differ from the oracle ({ref['kind']})"
    assert cb.bed_text(got["events"], ref["names"]) == ref["bed"]
    assert got["counters"] == ref["counters"]
    g.close()


@pytest.mark.parametrize("name", ["tiny", "c1s", "c2s", "c4s"])
@pytest.mark.parametrize("args", [["-9"], ["-1"], ["-3"], ["-5", "-q30"], ["-1", "-m10", "-C0.05", "-Z0.01"]], ids=lambda a: "".join(a))
def test_equals_process(name, args):
    batch = dataset(name)[2]
    n = int(batch.n_reads)
    rng = np.random.default_rng(len(name))
    check_cuts(batch, args, [every(n, 7), every(n, 1500), every(n, 20000), sorted(set(int(x) for x in rng.integers(0, n + 1, 12)))])


def test_deep_columns_cut_through():
    """VDEEP amplicons and STR triggers at depth, cut inside their deep columns"""
    data, nr, nb = cb.simulate("C4", 0.01, seed=9, amplicon_depth=16000, n_amplicons=2, threads=2)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    n = int(batch.n_reads)
    for args in (["-9"], ["-1"]):
        check_cuts(batch, args, [every(n, 4096), every(n, 1237)])
    bb.close()
    batch = dataset("c4m")[2]
    n = int(batch.n_reads)
    for args in (["-9", "-D300"], ["-1", "-D300", "-X0.2"]):
        check_cuts(batch, args, [every(n, 50000), every(n, 7777)])


@pytest.mark.parametrize("args", [["-9"], ["-1", "-B"]], ids=lambda a: "".join(a))
def test_full_size_c2(args):
    """whole synthetic chr20 (C2) in 1 Mi-record pushes: the same sha256 as process_device on the whole batch, and the held records stay
    below 10 000 after every push"""
    data, nr, nb = cb.simulate("C2", 1.0, seed=100)
    bb = cb.BatchBuilder(); bb.add_bam_stream(data); batch = bb.finish()
    del data
    g = cb.Crumble(params_from_opts(args, ["chr20"]), device=0)
    t = cb.device_batch(batch, 0)
    whole = g.process_device(t)
    ref_sha = hashlib.sha256(whole["qual"].cpu().numpy().tobytes()).hexdigest()
    got = stream_all(g, cb.split_device_batch(t, 1 << 20))
    assert hashlib.sha256(got["qual"].tobytes()).hexdigest() == ref_sha
    assert np.array_equal(got["events"], whole["events"]) and got["counters"] == whole["counters"]
    assert len(got["held"]) > 3 and max(got["held"]) < 10000, got["held"]
    g.close(); bb.close()


def test_non_default_stream_and_stream_check():
    """every push queued on a non-default stream behind a long sleep, nothing synchronised in between; a push from another stream is
    refused"""
    data, bb, batch, mask = dataset("c1s")
    g = cb.Crumble(params_from_opts(["-1"]), device=0)
    ref = g.process(batch); ref["qual"] = strip(batch, ref["qual"])
    t = cb.device_batch(batch, 0)
    chunks = cb.split_device_batch(t, 3001)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    outs = []
    with torch.cuda.stream(s):
        torch.cuda._sleep(200_000_000)
        st = g.device_stream()
        for ch in chunks:
            outs.append(st.push(dict(ch, qual=ch["qual"] + 0)))        # made by a kernel on this stream
        with torch.cuda.stream(torch.cuda.Stream()):
            with pytest.raises(cb.CrumbleError):
                st.push(chunks[0])
        outs.append(st.close())
    s.synchronize()
    assert np.array_equal(np.concatenate([o["qual"].cpu().numpy() for o in outs]), ref["qual"])
    g.close()


def test_one_chunk_buffer_reused_and_aliased_output():
    """every chunk copied into the same buffers, overwritten by the next chunk right after the call returns; then again with qual_out =
    the chunk's own quality buffer"""
    data, bb, batch, mask = dataset("c2s")
    g = cb.Crumble(params_from_opts(["-9"]), device=0)
    ref = g.process(batch); ref["qual"] = strip(batch, ref["qual"])
    t = cb.device_batch(batch, 0)
    chunks = cb.split_device_batch(t, 2000)
    big = {k: torch.empty(max(int(sum(c[k].numel() for c in chunks)), 1) + (1 << 20), dtype=v.dtype, device="cuda") for k, v in t.items()}
    for alias in (False, True):
        st = g.device_stream()
        q = []
        for ch in chunks:
            view = {k: big[k][: ch[k].numel()] for k in ch}
            for k in ch:
                view[k].copy_(ch[k])
            r = st.push(view, out=big["qual"] if alias else None)
            q.append(r["qual"].clone())                                 # queued before the next chunk overwrites the buffer
        q.append(st.close()["qual"].clone())
        assert np.array_equal(torch.cat(q).cpu().numpy(), ref["qual"]), f"alias {alias}"
    g.close()


def test_events_refetched_and_calls_refused_while_open():
    data, bb, batch, mask = dataset("tiny")
    g = cb.Crumble(params_from_opts(["-1"]), device=0)
    ref = g.process(batch); ref["qual"] = strip(batch, ref["qual"])
    t = cb.device_batch(batch, 0)
    chunks = cb.split_device_batch(t, 500)
    got = stream_all(g, chunks, events_cap=1)
    assert_same(ref, got, "events_cap=1")
    st = g.device_stream()
    st.push(chunks[0])
    for call in (lambda: g.process(batch), lambda: g.process_device(t), lambda: g.upload(batch), lambda: g.run(),
                 lambda: g.set_stream(torch.cuda.current_stream().cuda_stream), lambda: g.device_stream()):
        with pytest.raises(cb.CrumbleError):
            call()
    for ch in chunks[1:]:
        st.push(ch)
    st.close()
    r = g.process(batch)                                                # the context is free again
    assert np.array_equal(strip(batch, r["qual"]), ref["qual"])
    g.close()
