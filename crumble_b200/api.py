"""ctypes binding of the C ABI in include/crumble_gpu.h (libcrumble_gpu.so).

Host-side mirror of the reference interface for the hot path: the option block
(cram_lossy_params, reference snp_score.c:185-226), the level presets (2380-2482) and
``transcode`` (1336-2029) expressed as ``Crumble.process(batch)``.

There is no CPU fallback: if the shared library is missing, or no CUDA device is
usable, every compute call raises.  PyTorch is only imported by the device-resident entries
(``device_batch``, ``Crumble.process_device``, ``DeviceStream``); everything else works without it.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_DIR = _HERE / "lib"
N_COUNTERS = 19
COUNTER_NAMES = [
    "diff", "indel_qual", "indel", "het_qual_A", "het_A", "hom_qual_A", "hom_A", "discrep_A",
    "het_qual_B", "het_B", "hom_qual_B", "hom_B", "discrep_B", "columns", "low_mqual_perc",
    "clip_perc", "ins_len_perc", "indel_ov_perc", "over_depth",
]
BED_TAGS = ["VDEEP", "DEEP", "CLIP", "INDEL_LEN", "INDEL_COVERAGE"]
TIMERS = ["total", "tiles", "columns", "flagged", "depth", "chain", "rewrite", "cells", "events", "h2d", "d2h"]


class CrumbleError(RuntimeError):
    pass


class BedReg(C.Structure):
    _fields_ = [("tid", C.c_int32), ("start", C.c_int32), ("end", C.c_int32)]


class Params(C.Structure):
    """cg_params: POD mirror of cram_lossy_params."""
    _fields_ = [
        ("reduce_qual", C.c_int32), ("binary_qual", C.c_int32),
        ("iSTR_add", C.c_int32), ("sSTR_add", C.c_int32),
        ("iSTR_mul", C.c_double), ("sSTR_mul", C.c_double),
        ("qlow", C.c_int32), ("qcutoff", C.c_int32), ("qhigh", C.c_int32), ("qcap", C.c_int32),
        ("min_mqual", C.c_int32),
        ("indel_fract", C.c_double),
        ("min_qual_A", C.c_int32), ("min_indel_A", C.c_int32), ("min_discrep_A", C.c_double),
        ("min_qual_B", C.c_int32), ("min_indel_B", C.c_int32), ("min_discrep_B", C.c_double),
        ("low_mqual_perc", C.c_double), ("clip_perc", C.c_double), ("ins_len_perc", C.c_double),
        ("over_depth", C.c_double), ("indel_ov_perc", C.c_double),
        ("pblock", C.c_int32), ("softclip", C.c_int32), ("perfect_col", C.c_int32),
        ("verbose", C.c_int32), ("noPG", C.c_int32),
        ("region_tid", C.c_int32), ("region_beg", C.c_int32), ("region_end", C.c_int32),
        ("preserve_qual", C.c_uint8 * 256),
        ("bed", C.POINTER(BedReg)), ("nbed", C.c_int32),
    ]


class Batch(C.Structure):
    _fields_ = [
        ("n_reads", C.c_int64),
        ("tid", C.POINTER(C.c_int32)), ("pos", C.POINTER(C.c_int32)), ("flag", C.POINTER(C.c_uint16)),
        ("mapq", C.POINTER(C.c_uint8)), ("l_qseq", C.POINTER(C.c_int32)), ("n_cigar", C.POINTER(C.c_uint16)),
        ("off", C.POINTER(C.c_int64)), ("cigar_off", C.POINTER(C.c_int32)),
        ("cigar", C.POINTER(C.c_uint32)), ("n_cigar_total", C.c_int64),
        ("seq", C.POINTER(C.c_uint8)), ("seq_bytes", C.c_int64),
        ("qual", C.POINTER(C.c_uint8)), ("qual_bytes", C.c_int64),
        ("packed", C.c_int32),
        ("seq2", C.POINTER(C.c_uint8)), ("seq2_bytes", C.c_int64),
        ("seq_exc", C.POINTER(C.c_uint64)), ("n_seq_exc", C.c_int64),
        ("qualp", C.POINTER(C.c_uint8)), ("qualp_bytes", C.c_int64),
        ("qual_bits", C.c_int32), ("qual_dict", C.c_uint8 * 16),
        ("pmax_end", C.POINTER(C.c_int32)),
        ("meta_planes", C.c_int32),
        ("tid_runs", C.POINTER(C.c_uint64)), ("n_tid_runs", C.c_int64),
        ("pos_d8", C.POINTER(C.c_uint8)),
        ("pos_abs", C.POINTER(C.c_uint64)), ("n_pos_abs", C.c_int64),
        ("lq8", C.POINTER(C.c_uint8)), ("lq_dict", C.c_int32 * 256),
        ("nc8", C.POINTER(C.c_uint8)),
        ("cigar_x", C.POINTER(C.c_uint32)), ("n_cigar_x", C.c_int64),
    ]


class DevBatch(C.Structure):
    """cg_dev_batch: records already in GPU memory as concatenated BAM fields (include/crumble_gpu.h)."""
    _fields_ = [
        ("n_reads", C.c_int64),
        ("tid", C.c_void_p), ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p),
        ("l_qseq", C.c_void_p), ("n_cigar", C.c_void_p),
        ("cigar", C.c_void_p), ("n_cigar_total", C.c_int64),
        ("seq", C.c_void_p), ("seq_len", C.c_int64),
        ("qual", C.c_void_p), ("qual_len", C.c_int64),
    ]


# the arrays of a cg_dev_batch, their numpy dtypes, and which of them hold one entry per record
DEV_FIELDS = {"tid": np.int32, "pos": np.int32, "flag": np.uint16, "mapq": np.uint8, "l_qseq": np.int32, "n_cigar": np.uint16,
              "cigar": np.uint32, "seq": np.uint8, "qual": np.uint8}
DEV_PER_RECORD = ("tid", "pos", "flag", "mapq", "l_qseq", "n_cigar")


class StreamOut(C.Structure):
    """cg_stream_out: what one call of a stream of device records emitted and what the context still holds (include/crumble_gpu.h)."""
    _fields_ = [("n_records", C.c_int64), ("qual_len", C.c_int64), ("held_records", C.c_int64), ("held_qual_len", C.c_int64)]


class BedEvent(C.Structure):
    _fields_ = [("tid", C.c_int32), ("pos", C.c_int32), ("tag", C.c_int32)]


class Column(C.Structure):
    _fields_ = [("tid", C.c_int32), ("pos", C.c_int32), ("n_plp", C.c_int32), ("call", C.c_int32),
                ("het_call", C.c_int32), ("het_phred", C.c_int32), ("phred", C.c_int32),
                ("discrep", C.c_float), ("flags", C.c_uint32)]


COLUMN_DTYPE = np.dtype([("tid", "<i4"), ("pos", "<i4"), ("n_plp", "<i4"), ("call", "<i4"), ("het_call", "<i4"),
                         ("het_phred", "<i4"), ("phred", "<i4"), ("discrep", "<f4"), ("flags", "<u4")])
EVENT_DTYPE = np.dtype([("tid", "<i4"), ("pos", "<i4"), ("tag", "<i4")])


class Result(C.Structure):
    _fields_ = [
        ("qual_out", C.POINTER(C.c_uint8)),
        ("events", C.POINTER(BedEvent)), ("events_cap", C.c_int64), ("n_events", C.c_int64),
        ("counters", C.c_int64 * N_COUNTERS),
        ("columns", C.POINTER(Column)), ("columns_cap", C.c_int64), ("n_columns", C.c_int64),
        ("qual_head", C.POINTER(C.c_uint8)), ("head_bytes", C.c_int64),
    ]


class Window(C.Structure):
    """cg_window: the reference columns one call of a chain owns (include/crumble_gpu.h)."""
    _fields_ = [("first", C.c_int32), ("lo_tid", C.c_int32), ("lo_pos", C.c_int32), ("cnt_pos", C.c_int32),
                ("hi_tid", C.c_int32), ("hi_pos", C.c_int32), ("next_lo_pos", C.c_int32)]


_lib = None
_sim = None

EXPORTS = [
    "cg_abi_version", "cg_device_count", "cg_create", "cg_destroy", "cg_set_params", "cg_strerror", "cg_last_error",
    "cg_set_stream", "cg_process", "cg_process_device", "cg_stream_device", "cg_process_window", "cg_upload", "cg_run", "cg_download", "cg_sync", "cg_last_ms", "cg_last_launches", "cg_last_h2d_bytes",
    "cg_algorithmic_bytes", "cg_aligned_bases", "cg_n_columns", "cg_params_default", "cg_params_level",
    "cgb_create", "cgb_destroy", "cgb_reset", "cgb_add", "cgb_add_bam_stream", "cgb_finish", "cgb_bytes", "cgb_reserve", "cgb_pack",
    "cg_carry_export", "cg_carry_import", "cg_carry_is_neutral", "cg_batch_ends", "cg_shard_begin", "cg_shard_carry", "cg_shard_end",
    "cgm_create", "cgm_destroy", "cgm_n_devices", "cgm_process", "cgm_process_window", "cgm_last_error", "cgm_last_ms", "cgm_last_h2d_bytes", "cgm_context", "cgm_events",
]
CARRY_BYTES = 128


def lib_path() -> Path:
    # CRUMBLE_GPU_LIB: A/B runs of differently tuned builds of the same library (tools/build_variant.sh)
    return Path(os.environ["CRUMBLE_GPU_LIB"]) if os.environ.get("CRUMBLE_GPU_LIB") else LIB_DIR / "libcrumble_gpu.so"


def load_lib():
    """Load libcrumble_gpu.so (built in-tree by ``__graft_entry__.build()``); raise loudly if absent."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not p.exists():
        raise CrumbleError(f"{p} is missing: the CUDA extension is mandatory (run `python -c 'import __graft_entry__ as g; g.build()'`)")
    lib = C.CDLL(str(p))
    lib.cg_abi_version.restype = C.c_int
    lib.cg_device_count.restype = C.c_int
    lib.cg_create.restype = C.c_void_p
    lib.cg_create.argtypes = [C.POINTER(Params), C.c_int, C.POINTER(C.c_int)]
    lib.cg_destroy.argtypes = [C.c_void_p]
    lib.cg_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
    lib.cg_strerror.restype = C.c_char_p
    lib.cg_strerror.argtypes = [C.c_int]
    lib.cg_last_error.restype = C.c_char_p
    lib.cg_last_error.argtypes = [C.c_void_p]
    lib.cg_set_stream.argtypes = [C.c_void_p, C.c_void_p]
    for f in ("cg_process",):
        getattr(lib, f).argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Result)]
    lib.cg_process_window.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Window), C.POINTER(Result)]
    lib.cg_process_device.argtypes = [C.c_void_p, C.POINTER(DevBatch), C.c_void_p, C.POINTER(Result)]
    lib.cg_stream_device.argtypes = [C.c_void_p, C.POINTER(DevBatch), C.c_int, C.c_void_p, C.c_int64, C.POINTER(Result), C.POINTER(StreamOut)]
    lib.cgb_reserve.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64]
    lib.cg_carry_export.argtypes = [C.c_void_p, C.c_void_p]
    lib.cg_carry_import.argtypes = [C.c_void_p, C.c_void_p]
    lib.cg_carry_is_neutral.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]
    lib.cg_batch_ends.argtypes = [C.POINTER(Batch), C.c_void_p]
    lib.cg_shard_begin.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Window), C.POINTER(Result)]
    lib.cg_shard_carry.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cg_shard_end.argtypes = [C.c_void_p, C.POINTER(Result)]
    lib.cgm_create.restype = C.c_void_p
    lib.cgm_create.argtypes = [C.POINTER(Params), C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.cgm_destroy.argtypes = [C.c_void_p]
    lib.cgm_n_devices.argtypes = [C.c_void_p]
    lib.cgm_process.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Result)]
    lib.cgm_process_window.argtypes = [C.c_void_p, C.POINTER(Batch), C.POINTER(Window), C.POINTER(Result)]
    lib.cgm_last_error.restype = C.c_char_p
    lib.cgm_last_error.argtypes = [C.c_void_p]
    lib.cgm_last_ms.restype = C.c_float
    lib.cgm_last_ms.argtypes = [C.c_void_p]
    lib.cgm_last_h2d_bytes.restype = C.c_int64
    lib.cgm_last_h2d_bytes.argtypes = [C.c_void_p]
    lib.cg_upload.argtypes = [C.c_void_p, C.POINTER(Batch)]
    lib.cg_run.argtypes = [C.c_void_p]
    lib.cg_sync.argtypes = [C.c_void_p]
    lib.cg_set_chunk_bytes.argtypes = [C.c_void_p, C.c_int64]
    lib.cg_download.argtypes = [C.c_void_p, C.POINTER(Result)]
    lib.cg_last_ms.restype = C.c_float
    lib.cg_last_ms.argtypes = [C.c_void_p, C.c_int]
    lib.cg_last_launches.restype = C.c_int64
    lib.cg_last_launches.argtypes = [C.c_void_p]
    lib.cg_last_h2d_bytes.restype = C.c_int64
    lib.cg_last_h2d_bytes.argtypes = [C.c_void_p]
    lib.cg_n_columns.restype = C.c_int64
    lib.cg_n_columns.argtypes = [C.c_void_p]
    lib.cg_algorithmic_bytes.restype = C.c_int64
    lib.cg_algorithmic_bytes.argtypes = [C.POINTER(Batch)]
    lib.cg_aligned_bases.restype = C.c_int64
    lib.cg_aligned_bases.argtypes = [C.POINTER(Batch)]
    lib.cg_params_default.argtypes = [C.POINTER(Params)]
    lib.cg_params_level.argtypes = [C.POINTER(Params), C.c_int]
    lib.cgb_create.restype = C.c_void_p
    lib.cgb_create.argtypes = [C.c_int]
    lib.cgb_destroy.argtypes = [C.c_void_p]
    lib.cgb_reset.argtypes = [C.c_void_p]
    lib.cgb_add_bam_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
    lib.cgb_add.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_uint16, C.c_uint8, C.c_int32, C.c_uint32,
                            C.c_void_p, C.c_void_p, C.c_void_p]
    lib.cgb_finish.argtypes = [C.c_void_p, C.POINTER(Batch)]
    lib.cgb_pack.argtypes = [C.c_void_p, C.c_int]
    lib.cgb_bytes.restype = C.c_int64
    lib.cgb_bytes.argtypes = [C.c_void_p]
    lib.crumble_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    _lib = lib
    return lib


def _check(lib, code, ctx=None):
    if code != 0:
        detail = lib.cg_last_error(ctx).decode() if ctx else ""
        raise CrumbleError(f"{lib.cg_strerror(code).decode()} [{code}] {detail}")


def default_params(level: int | None = None, **overrides) -> Params:
    """Reference defaults (snp_score.c:2152-2192), optionally a level preset, then field overrides."""
    lib = load_lib()
    p = Params()
    lib.cg_params_default(C.byref(p))
    if level is not None:
        _check(lib, lib.cg_params_level(C.byref(p), level))
    for k, v in overrides.items():
        setattr(p, k, v)
    return p


class BatchBuilder:
    """Host batcher: decoded records -> (pinned) structure-of-arrays."""

    def __init__(self, pinned: bool = True):
        self.lib = load_lib()
        self.h = self.lib.cgb_create(1 if pinned else 0)
        if not self.h:
            raise CrumbleError("cgb_create failed")
        self.batch = Batch()
        self._keep = []

    def add_bam_stream(self, buf: np.ndarray):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        _check(self.lib, self.lib.cgb_add_bam_stream(self.h, buf.ctypes.data, buf.size))

    def add(self, tid, pos, flag, mapq, cigar, seq4, qual):
        cigar = np.ascontiguousarray(cigar, dtype=np.uint32)
        seq4 = np.ascontiguousarray(seq4, dtype=np.uint8)
        qual = np.ascontiguousarray(qual, dtype=np.uint8)
        _check(self.lib, self.lib.cgb_add(self.h, tid, pos, flag, mapq, qual.size, cigar.size,
                                          cigar.ctypes.data, seq4.ctypes.data, qual.ctypes.data))

    def finish(self, pack: bool = False, threads: int = 0) -> Batch:
        """pack=True also builds the compact planes (2-bit bases + exception list, dictionary-coded qualities when the batch has at
        most 16 distinct values): the upload then moves those instead of seq / qual"""
        if pack:
            _check(self.lib, self.lib.cgb_pack(self.h, threads))
        _check(self.lib, self.lib.cgb_finish(self.h, C.byref(self.batch)))
        return self.batch

    def offsets(self) -> np.ndarray:
        n = self.batch.n_reads
        return np.ctypeslib.as_array(self.batch.off, shape=(n,)).copy() if n else np.zeros(0, np.int64)

    def positions(self) -> np.ndarray:
        n = self.batch.n_reads
        return np.ctypeslib.as_array(self.batch.pos, shape=(n,)).copy() if n else np.zeros(0, np.int32)

    def lengths(self) -> np.ndarray:
        n = self.batch.n_reads
        return np.ctypeslib.as_array(self.batch.l_qseq, shape=(n,)).copy() if n else np.zeros(0, np.int32)

    def qual(self) -> np.ndarray:
        return np.ctypeslib.as_array(self.batch.qual, shape=(self.batch.qual_bytes,))

    def close(self):
        if self.h:
            self.lib.cgb_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Crumble:
    """One GPU context (one per device / process)."""

    def __init__(self, params: Params | None = None, device: int = 0):
        self.lib = load_lib()
        if self.lib.cg_device_count() <= 0:
            raise CrumbleError("no usable CUDA device: the GPU path is mandatory, there is no CPU fallback")
        self.params = params if params is not None else default_params()
        self.device = device
        err = C.c_int(0)
        self.h = self.lib.cg_create(C.byref(self.params), device, C.byref(err))
        if not self.h:
            raise CrumbleError(f"cg_create failed: {self.lib.cg_strerror(err.value).decode()}")
        self._qout = None

    def set_stream(self, cuda_stream_ptr: int):
        _check(self.lib, self.lib.cg_set_stream(self.h, C.c_void_p(cuda_stream_ptr)), self.h)

    def _result(self, batch: Batch, want_columns: bool, events_cap: int, pinned_out=None):
        res = Result()
        if pinned_out is not None:
            qout = pinned_out
        else:
            qout = np.empty(max(int(batch.qual_bytes), 1), dtype=np.uint8)
        res.qual_out = qout.ctypes.data_as(C.POINTER(C.c_uint8))
        ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
        res.events = ev.ctypes.data_as(C.POINTER(BedEvent))
        res.events_cap = events_cap
        cols = None
        if want_columns:
            cap = int(getattr(self, "_ncols_hint", 0)) or 1
            cols = np.zeros(cap, dtype=COLUMN_DTYPE)
            res.columns = cols.ctypes.data_as(C.POINTER(Column))
            res.columns_cap = cap
        return res, qout, ev, cols

    def process(self, batch: Batch, want_columns: bool = False, events_cap: int = 1 << 16, pinned_out=None):
        """End to end: host SoA in, host results out (upload + kernel chain + download)."""
        if want_columns:
            # first pass sizes the dump
            self._ncols_hint = 1
        events_cap = max(events_cap, getattr(self, "_events_hint", 0))
        while True:
            res, qout, ev, cols = self._result(batch, want_columns, events_cap, pinned_out)
            _check(self.lib, self.lib.cg_process(self.h, C.byref(batch), C.byref(res)), self.h)
            if res.n_events > events_cap:                  # the list is still on the device: fetch it again, do not run the call twice
                events_cap = self._events_hint = int(res.n_events)
                n_cols, cols_cap = int(res.n_columns), int(res.columns_cap)
                res2, _, ev, _ = self._result(batch, False, events_cap, qout)
                res2.qual_out = None                       # the qualities are already home
                _check(self.lib, self.lib.cg_download(self.h, C.byref(res2)), self.h)
                res2.n_columns, res2.columns_cap = n_cols, cols_cap
                res = res2
            if want_columns and res.n_columns > res.columns_cap:
                self._ncols_hint = int(res.n_columns)
                continue
            break
        out = {
            "qual": qout[: int(batch.qual_bytes)],
            "events": ev[: int(res.n_events)],
            "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)},
        }
        if want_columns:
            out["columns"] = cols[: int(res.n_columns)]
        return out

    def process_device(self, tensors: dict, out=None, want_columns: bool = False, events_cap: int = 1 << 16):
        """Records already in GPU memory (cg_process_device): ``tensors`` holds the concatenated BAM fields of ``device_batch`` as
        contiguous 1-D tensors on this context's device; the rewritten qualities land in ``out`` (same layout, may be ``tensors["qual"]``
        itself) or in a new tensor from torch's caching allocator.  Runs on torch's current stream of the device, so work queued there
        before the call is its input and work queued after it sees the result.  Returns {"qual", "events", "counters"[, "columns"]}."""
        import torch
        dev = torch.device("cuda", self.device)
        t, db = self._dev_batch(tensors, "process_device")
        qual_len = t["qual"].numel()
        if out is None:
            out = torch.empty(qual_len, dtype=torch.uint8, device=dev)
        elif not isinstance(out, torch.Tensor) or out.device != dev or out.dtype != torch.uint8 or out.dim() != 1 or not out.is_contiguous() \
                or out.numel() != qual_len:
            raise CrumbleError(f"process_device: out must be a contiguous uint8 tensor of {qual_len} bytes on {dev}")
        self.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        events_cap = max(events_cap, getattr(self, "_events_hint", 0))
        ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
        res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=events_cap)
        cols = None
        if want_columns:
            cap = int(getattr(self, "_ncols_hint", 0)) or 1
            cols = np.zeros(cap, dtype=COLUMN_DTYPE)
            res.columns, res.columns_cap = cols.ctypes.data_as(C.POINTER(Column)), cap
        _check(self.lib, self.lib.cg_process_device(self.h, C.byref(db), out.data_ptr() or None, C.byref(res)), self.h)
        if res.n_events > events_cap or (want_columns and res.n_columns > res.columns_cap):
            # still on the device: fetch again with room for everything; the call is not repeated (it may have rewritten in place)
            if res.n_events > events_cap:
                events_cap = self._events_hint = int(res.n_events)
                ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
            res2 = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=events_cap)
            if want_columns:
                if res.n_columns > res.columns_cap:
                    self._ncols_hint = int(res.n_columns)
                    cols = np.zeros(self._ncols_hint, dtype=COLUMN_DTYPE)
                res2.columns, res2.columns_cap = cols.ctypes.data_as(C.POINTER(Column)), len(cols)
            _check(self.lib, self.lib.cg_download(self.h, C.byref(res2)), self.h)
            res = res2
        r = {"qual": out, "events": ev[: int(res.n_events)], "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}}
        if want_columns:
            r["columns"] = cols[: int(res.n_columns)]
        return r

    def _dev_batch(self, tensors: dict, what: str):
        """the checked tensors of a device_batch dict and the cg_dev_batch over them"""
        import torch
        dev = torch.device("cuda", self.device)
        t = {}
        for k, dt in DEV_FIELDS.items():
            x = tensors.get(k)
            if not isinstance(x, torch.Tensor):
                raise CrumbleError(f"{what}: {k} must be a torch tensor")
            if x.device != dev:
                raise CrumbleError(f"{what}: {k} is on {x.device}, the context runs on {dev}")
            if x.dtype != _torch_dtype(dt):
                raise CrumbleError(f"{what}: {k} must be {_torch_dtype(dt)}, not {x.dtype}")
            if x.dim() != 1 or not x.is_contiguous():
                raise CrumbleError(f"{what}: {k} must be a contiguous 1-D tensor")
            t[k] = x
        n = t["tid"].numel()
        for k in DEV_PER_RECORD:
            if t[k].numel() != n:
                raise CrumbleError(f"{what}: {k} has {t[k].numel()} entries, tid has {n}: one per record")
        db = DevBatch(n_reads=n, n_cigar_total=t["cigar"].numel(), seq_len=t["seq"].numel(), qual_len=t["qual"].numel())
        for k in DEV_FIELDS:
            setattr(db, k, t[k].data_ptr() or None)
        return t, db

    def device_stream(self) -> "DeviceStream":
        """A coordinate-sorted stream of device records pushed in chunks of any size (cg_stream_device); see ``DeviceStream``."""
        if getattr(self, "_stream", None) is not None and not self._stream.closed:
            raise CrumbleError("device_stream: a stream is already open on this context")
        self._stream = DeviceStream(self)
        return self._stream

    def process_window(self, batch: Batch, window: Window, events_cap: int = 1 << 16, pinned_out=None):
        """One call of a chain (cg_process_window): ``batch`` = read halo + new records, ``window`` = the columns it owns.
        The keep-window and depth-average state stay inside the context between calls."""
        res, qout, ev, _ = self._result(batch, False, events_cap, pinned_out)
        _check(self.lib, self.lib.cg_process_window(self.h, C.byref(batch), C.byref(window), C.byref(res)), self.h)
        if res.n_events > events_cap:                      # the chain's state has moved on: fetch again, do not redo
            res, qout, ev, _ = self._result(batch, False, int(res.n_events), pinned_out)
            _check(self.lib, self.lib.cg_download(self.h, C.byref(res)), self.h)
        return {"qual": qout[: int(batch.qual_bytes)], "events": ev[: int(res.n_events)],
                "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}}

    # region shards without speculation: begin (state-free part) on all shards, carry from left to right, end on all shards
    def shard_begin(self, batch: Batch | None, window: Window, events_cap: int = 1 << 16, pinned_out=None):
        """batch None: the batch ``upload`` left on the device (the chain alone, no copies: what bench.py times as `value`)"""
        if batch is None:
            res = Result(); ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
            res.events = ev.ctypes.data_as(C.POINTER(BedEvent)); res.events_cap = events_cap
            self._shard = (None, (res, None, ev, None))
            _check(self.lib, self.lib.cg_shard_begin(self.h, None, C.byref(window), C.byref(res)), self.h)
            return
        self._shard = (batch, self._result(batch, False, events_cap, pinned_out))
        _check(self.lib, self.lib.cg_shard_begin(self.h, C.byref(batch), C.byref(window), C.byref(self._shard[1][0])), self.h)

    def shard_carry(self, carry_in: bytes | None, want_out: bool = True) -> bytes | None:
        cin = C.create_string_buffer(carry_in, CARRY_BYTES) if carry_in is not None else None
        cout = C.create_string_buffer(CARRY_BYTES) if want_out else None
        _check(self.lib, self.lib.cg_shard_carry(self.h, cin, cout), self.h)
        return cout.raw if want_out else None

    def shard_end(self):
        batch, (res, qout, ev, _) = self._shard
        _check(self.lib, self.lib.cg_shard_end(self.h, C.byref(res)), self.h)
        if batch is None:
            self._shard = None
            return {"qual": None, "events": ev[: min(int(res.n_events), int(res.events_cap))], "n_events": int(res.n_events),
                    "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}}
        if res.n_events > res.events_cap:
            res2, qout2, ev, _ = self._result(batch, False, int(res.n_events), qout)
            _check(self.lib, self.lib.cg_download(self.h, C.byref(res2)), self.h)
            res = res2
        self._shard = None
        return {"qual": qout[: int(batch.qual_bytes)], "events": ev[: int(res.n_events)],
                "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}}

    def carry_export(self) -> bytes:
        """the cross-column state the last ``process_window`` saved at its ``next_lo_pos`` (opaque, CARRY_BYTES long)"""
        buf = C.create_string_buffer(CARRY_BYTES)
        _check(self.lib, self.lib.cg_carry_export(self.h, buf), self.h)
        return buf.raw

    def carry_import(self, blob: bytes):
        _check(self.lib, self.lib.cg_carry_import(self.h, C.create_string_buffer(blob, CARRY_BYTES)), self.h)

    def carry_is_neutral(self, blob: bytes, tid: int, lo_pos: int) -> int:
        """1 neutral, 0 open keep window (re-run this shard from blob), -1 depth average in play (re-run the chain in order)"""
        return int(self.lib.cg_carry_is_neutral(self.h, C.create_string_buffer(blob, CARRY_BYTES), tid, lo_pos))

    # split phase (resident timing)
    def set_chunk_bytes(self, nbytes: int):
        """Upload-chunk size of the streamed ``process`` (results do not depend on it)."""
        _check(self.lib, self.lib.cg_set_chunk_bytes(self.h, int(nbytes)), self.h)

    def upload(self, batch: Batch):
        _check(self.lib, self.lib.cg_upload(self.h, C.byref(batch)), self.h)

    def run(self):
        _check(self.lib, self.lib.cg_run(self.h), self.h)

    def download(self, batch: Batch, events_cap: int = 1 << 16, pinned_out=None):
        res, qout, ev, _ = self._result(batch, False, events_cap, pinned_out)
        _check(self.lib, self.lib.cg_download(self.h, C.byref(res)), self.h)
        return {"qual": qout[: int(batch.qual_bytes)], "events": ev[: min(int(res.n_events), events_cap)],
                "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}, "n_events": int(res.n_events)}

    def ms(self, which: str = "total") -> float:
        return float(self.lib.cg_last_ms(self.h, TIMERS.index(which)))

    def timers(self) -> dict:
        return {k: self.ms(k) for k in TIMERS}

    def h2d_bytes(self) -> int:
        return int(self.lib.cg_last_h2d_bytes(self.h))

    def launches(self) -> int:
        return int(self.lib.cg_last_launches(self.h))

    def n_columns(self) -> int:
        return int(self.lib.cg_n_columns(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.cg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class DeviceStream:
    """One stream of records in GPU memory on a context (cg_stream_device).  ``push(tensors)`` appends the next records of the stream (a
    ``device_batch`` dict, or a chunk of one from ``split_device_batch``) and returns the rewritten qualities of the records that became
    final, in stream order: {"qual": uint8 CUDA tensor, "n_records", "events", "counters", "held_records"}.  ``close()`` ends the stream
    and returns the rest the same way.  The concatenated qualities and events and the summed counters of all calls equal one
    ``process_device`` on the whole stream.  Every call runs on the torch stream that was current at the first push."""

    def __init__(self, g: Crumble):
        self.g = g
        self.stream = None
        self.held_qual_len = 0
        self.closed = False

    def push(self, tensors: dict | None, events_cap: int = 1 << 16, last: bool = False, out=None):
        """``out``: a contiguous uint8 CUDA tensor of at least held + new quality bytes (may be ``tensors["qual"]``); by default a new one"""
        import torch
        g = self.g
        if self.closed:
            raise CrumbleError("push: the stream is closed")
        if g.params.region_tid >= 0:
            raise CrumbleError("push: streams and a -r region do not combine")
        dev = torch.device("cuda", g.device)
        cur = torch.cuda.current_stream(dev)
        if self.stream is None:
            g.set_stream(cur.cuda_stream)
            self.stream = cur
        elif cur.cuda_stream != self.stream.cuda_stream:
            raise CrumbleError("push: the current torch stream is not the one the stream started on")
        if tensors is None:
            db, new_len, keep = None, 0, None
        else:
            keep, db = g._dev_batch(tensors, "push")
            new_len = int(db.qual_len)
        cap = self.held_qual_len + new_len
        if out is None:
            out = torch.empty(max(cap, 1), dtype=torch.uint8, device=dev)
        elif not isinstance(out, torch.Tensor) or out.device != dev or out.dtype != torch.uint8 or out.dim() != 1 or not out.is_contiguous() \
                or out.numel() < cap:
            raise CrumbleError(f"push: out must be a contiguous uint8 tensor of at least {cap} bytes on {dev}")
        events_cap = max(events_cap, 1)
        ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
        res = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=events_cap)
        so = StreamOut()
        code = g.lib.cg_stream_device(g.h, C.byref(db) if db is not None else None, 1 if last else 0, out.data_ptr(), out.numel(), C.byref(res), C.byref(so))
        if code != 0:
            self.closed = True                             # what this class checks up front cannot fail in C: the rest closes the stream
            g._stream = None
        _check(g.lib, code, g.h)
        if res.n_events > events_cap:                      # the chain's state has moved on: fetch the list again, do not redo
            ev = np.zeros(int(res.n_events), dtype=EVENT_DTYPE)
            res2 = Result(events=ev.ctypes.data_as(C.POINTER(BedEvent)), events_cap=int(res.n_events))
            _check(g.lib, g.lib.cg_download(g.h, C.byref(res2)), g.h)
            res = res2
        self.held_qual_len = int(so.held_qual_len)
        if last:
            self.closed = True
            g._stream = None
        return {"qual": out[: int(so.qual_len)], "n_records": int(so.n_records), "events": ev[: int(res.n_events)],
                "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}, "held_records": int(so.held_records)}

    def close(self, events_cap: int = 1 << 16):
        """the last call: everything the context still holds comes out, and the stream ends"""
        return self.push(None, events_cap=events_cap, last=True)


class MultiCrumble:
    """cg_multi: one batch over several devices (region shards scheduled in C, crumble_b200/csrc/cg_multi.c).  ``devices`` may name a
    device more than once (several contexts on one GPU)."""

    def __init__(self, params: Params | None = None, devices=None):
        self.lib = load_lib()
        if self.lib.cg_device_count() <= 0:
            raise CrumbleError("no usable CUDA device: the GPU path is mandatory, there is no CPU fallback")
        self.params = params if params is not None else default_params()
        err = C.c_int(0)
        if devices is None:
            self.h = self.lib.cgm_create(C.byref(self.params), 0, None, C.byref(err))
        else:
            arr = (C.c_int * len(devices))(*devices)
            self.h = self.lib.cgm_create(C.byref(self.params), len(devices), arr, C.byref(err))
        if not self.h:
            raise CrumbleError(f"cgm_create failed: {self.lib.cg_strerror(err.value).decode()}")

    def n_devices(self) -> int:
        return int(self.lib.cgm_n_devices(self.h))

    def process(self, batch: Batch, events_cap: int = 1 << 16, pinned_out=None, window: Window | None = None):
        events_cap = max(events_cap, getattr(self, "_events_hint", 0))
        while True:
            res = Result()
            qout = pinned_out if pinned_out is not None else np.empty(max(int(batch.qual_bytes), 1), dtype=np.uint8)
            res.qual_out = qout.ctypes.data_as(C.POINTER(C.c_uint8))
            ev = np.zeros(events_cap, dtype=EVENT_DTYPE)
            res.events = ev.ctypes.data_as(C.POINTER(BedEvent)); res.events_cap = events_cap
            code = self.lib.cgm_process(self.h, C.byref(batch), C.byref(res)) if window is None else \
                self.lib.cgm_process_window(self.h, C.byref(batch), C.byref(window), C.byref(res))
            if code != 0:
                raise CrumbleError(f"{self.lib.cg_strerror(code).decode()} [{code}] {self.lib.cgm_last_error(self.h).decode()}")
            if res.n_events > events_cap and window is None:
                events_cap = self._events_hint = int(res.n_events); continue
            break
        return {"qual": qout[: int(batch.qual_bytes)], "events": ev[: min(int(res.n_events), events_cap)], "n_events": int(res.n_events),
                "counters": {k: int(res.counters[i]) for i, k in enumerate(COUNTER_NAMES)}}

    def ms(self) -> float:
        return float(self.lib.cgm_last_ms(self.h))

    def h2d_bytes(self) -> int:
        return int(self.lib.cgm_last_h2d_bytes(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.cgm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def batch_ends(batch: Batch) -> np.ndarray:
    """pos + reference span of every record (pos itself outside the pileup): cg_batch_ends"""
    out = np.empty(int(batch.n_reads), dtype=np.int32)
    load_lib().cg_batch_ends(C.byref(batch), out.ctypes.data)
    return out


def sub_batch(batch: Batch, i0: int, i1: int):
    """Records [i0, i1) of a batch as a batch of their own: the big arrays are shared, the two offset arrays rebased.
    Returns (Batch, keepalive)."""
    n_all = int(batch.n_reads)
    off = np.ctypeslib.as_array(batch.off, shape=(n_all,))
    coff = np.ctypeslib.as_array(batch.cigar_off, shape=(n_all,))
    q0 = int(off[i0]); q1 = int(off[i1]) if i1 < n_all else int(batch.qual_bytes)
    c0 = int(coff[i0]); c1 = int(coff[i1]) if i1 < n_all else int(batch.n_cigar_total)
    off2 = (off[i0:i1] - q0).astype(np.int64); coff2 = (coff[i0:i1] - c0).astype(np.int32)

    def at(ptr, ctype, idx):
        return C.cast(C.addressof(ptr.contents) + C.sizeof(ctype) * idx, C.POINTER(ctype))
    b = Batch()
    b.n_reads = i1 - i0
    b.tid = at(batch.tid, C.c_int32, i0); b.pos = at(batch.pos, C.c_int32, i0); b.flag = at(batch.flag, C.c_uint16, i0)
    b.mapq = at(batch.mapq, C.c_uint8, i0); b.l_qseq = at(batch.l_qseq, C.c_int32, i0); b.n_cigar = at(batch.n_cigar, C.c_uint16, i0)
    b.off = off2.ctypes.data_as(C.POINTER(C.c_int64)); b.cigar_off = coff2.ctypes.data_as(C.POINTER(C.c_int32))
    b.cigar = at(batch.cigar, C.c_uint32, c0); b.n_cigar_total = c1 - c0
    b.seq = at(batch.seq, C.c_uint8, q0 // 2); b.seq_bytes = (q1 - q0) // 2
    b.qual = at(batch.qual, C.c_uint8, q0); b.qual_bytes = q1 - q0
    b.packed = batch.packed                            # running sums stay running sums after rebasing
    keep = [off2, coff2]
    if batch.seq2:                                     # compact planes: positions are quality-buffer offsets, so they rebase with q0
        b.seq2 = at(batch.seq2, C.c_uint8, q0 // 4); b.seq2_bytes = (q1 - q0) // 4
        ne = int(batch.n_seq_exc)
        exc = np.ctypeslib.as_array(batch.seq_exc, shape=(ne,)) if ne else np.zeros(0, np.uint64)
        e0, e1 = np.searchsorted(exc >> np.uint64(4), [q0, q1]) if ne else (0, 0)
        exc2 = (exc[e0:e1] - np.uint64(q0 << 4)).astype(np.uint64)
        keep.append(exc2)
        b.seq_exc = exc2.ctypes.data_as(C.POINTER(C.c_uint64)) if exc2.size else None
        b.n_seq_exc = int(exc2.size)
        b.qual_bits = batch.qual_bits
        if batch.qual_bits:
            b.qualp = at(batch.qualp, C.c_uint8, q0 * batch.qual_bits // 8); b.qualp_bytes = (q1 - q0) * batch.qual_bits // 8
            for k in range(16):
                b.qual_dict[k] = batch.qual_dict[k]
    return b, tuple(keep)


def _torch_dtype(np_dtype):
    import torch
    return {np.int32: torch.int32, np.uint16: torch.uint16, np.uint8: torch.uint8, np.uint32: torch.uint32}[np_dtype]


def _strip(buf: np.ndarray, off: np.ndarray, ln: np.ndarray, unit: int, packed: bool) -> np.ndarray:
    """bytes [off[i], off[i] + ln[i]) of every record, back to back.  A packed batch lays records out in whole rows of `unit` bytes with
    the padding at the end of each record's last row: a row mask strips it without an index per byte."""
    total = int(ln.sum())
    if total == 0:
        return buf[:0].copy()
    if packed and buf.size % unit == 0:
        rows = (ln + unit - 1) // unit
        keep = np.full(buf.size // unit, unit, np.uint8)
        has = rows > 0
        keep[(off[has] // unit + rows[has] - 1)] = (ln[has] - unit * (rows[has] - 1)).astype(np.uint8)
        return buf.reshape(-1, unit)[np.arange(unit, dtype=np.uint8)[None, :] < keep[:, None]]
    start = np.cumsum(ln) - ln
    return buf[np.arange(total, dtype=np.int64) + np.repeat(off - start, ln)]


def concat_fields(batch: Batch) -> dict:
    """A host Batch (from BatchBuilder) as the concatenated BAM fields of cg_dev_batch, in numpy: the per-record arrays as they are,
    the CIGARs, sequences (ceil(l/2) bytes) and qualities (l bytes) of the records back to back without the batcher's padding."""
    n = int(batch.n_reads)

    def arr(ptr, dtype, count):
        return np.ctypeslib.as_array(ptr, shape=(count,)).astype(dtype, copy=True) if count else np.zeros(0, dtype)
    f = {k: arr(getattr(batch, k), DEV_FIELDS[k], n) for k in DEV_PER_RECORD}
    ln = f["l_qseq"].astype(np.int64)
    off = arr(batch.off, np.int64, n)
    packed = batch.packed == 1
    cig = arr(batch.cigar, np.uint32, int(batch.n_cigar_total))
    f["cigar"] = _strip(cig, arr(batch.cigar_off, np.int64, n), f["n_cigar"].astype(np.int64), 1, False) if not packed else cig
    f["seq"] = _strip(np.ctypeslib.as_array(batch.seq, shape=(int(batch.seq_bytes),)) if batch.seq_bytes else np.zeros(0, np.uint8),
                      off // 2, (ln + 1) // 2, 4, packed)
    f["qual"] = _strip(np.ctypeslib.as_array(batch.qual, shape=(int(batch.qual_bytes),)) if batch.qual_bytes else np.zeros(0, np.uint8),
                       off, ln, 8, packed)
    return f


def device_batch(batch: Batch, device) -> dict:
    """The records of a host Batch as torch tensors on `device` (an index or a torch.device) in the layout ``Crumble.process_device``
    takes: what a GPU-side BAM decoder would hand over."""
    import torch
    dev = torch.device("cuda", device) if isinstance(device, int) else torch.device(device)
    return {k: torch.from_numpy(v).to(dev) for k, v in concat_fields(batch).items()}


def split_device_batch(tensors: dict, n_per_chunk: int | None = None, cuts=None) -> list:
    """Cut a ``device_batch`` dict (torch tensors, or numpy arrays of the same layout) into consecutive chunk dicts, every
    ``n_per_chunk`` records or before each record index in ``cuts``.  The chunks are views of the input."""
    n = int(tensors["tid"].shape[0])
    if cuts is None:
        if not n_per_chunk or n_per_chunk < 1:
            raise CrumbleError("split_device_batch: give n_per_chunk >= 1 or cuts")
        cuts = range(n_per_chunk, n, n_per_chunk)
    b = [0] + sorted(int(c) for c in cuts) + [n]
    if b[1] < 0 or b[-2] > n:
        raise CrumbleError(f"split_device_batch: cuts must lie in [0, {n}]")
    host = lambda x: np.asarray(x.cpu()) if hasattr(x, "cpu") else np.asarray(x)
    lq, nc = host(tensors["l_qseq"]).astype(np.int64), host(tensors["n_cigar"]).astype(np.int64)
    q = np.concatenate([[0], np.cumsum(lq)]); s = np.concatenate([[0], np.cumsum((lq + 1) // 2)]); c = np.concatenate([[0], np.cumsum(nc)])
    chunks = []
    for i0, i1 in zip(b[:-1], b[1:]):
        d = {k: tensors[k][i0:i1] for k in DEV_PER_RECORD}
        d["cigar"] = tensors["cigar"][int(c[i0]):int(c[i1])]
        d["seq"] = tensors["seq"][int(s[i0]):int(s[i1])]
        d["qual"] = tensors["qual"][int(q[i0]):int(q[i1])]
        chunks.append(d)
    return chunks


def plan_region_shards(batch: Batch, n_shards: int):
    """Cut a batch into n_shards region shards of about equal record counts, each with its read halo (DESIGN.md §3.4/§5).
    Returns a list of dicts: records [h0, r1) form the shard's batch (halo [h0, r0) + own records [r0, r1)), with the
    cg_window fields of the call.  A record is final in the first shard that holds it and whose right cut X it does not
    reach (end <= X), or that has no right cut on its contig."""
    n = int(batch.n_reads)
    pos = np.ctypeslib.as_array(batch.pos, shape=(n,))
    tid = np.ctypeslib.as_array(batch.tid, shape=(n,))
    end = batch_ends(batch)
    cuts = [0] + [int(round(n * k / n_shards)) for k in range(1, n_shards)] + [n]
    shards = []
    lo = None                                         # (tid, S, X) of the previous cut
    for k in range(n_shards):
        r0, r1 = cuts[k], cuts[k + 1]
        sh = {"r0": r0, "r1": r1, "first": 1 if lo is None else 2, "lo_tid": -1, "lo_pos": 0, "cnt_pos": 0, "h0": r0,
              "hi_tid": -1, "hi_pos": 0, "next_lo_pos": 0}
        if lo is not None:
            t, S, X = lo
            sh["lo_tid"], sh["lo_pos"], sh["cnt_pos"] = t, S, X
            same = tid[:r0] == t                                              # the halo: records of that contig reaching beyond S
            reach = np.nonzero(same & (end[:r0] > S))[0]
            sh["h0"] = int(reach[0]) if reach.size else r0
        lo = None
        if r1 < n and r1 > 0 and tid[r1] >= 0 and tid[r1] == tid[r1 - 1]:
            t, X = int(tid[r1]), int(pos[r1])
            h = sh["h0"]
            open_ = np.nonzero((tid[h:r1] == t) & (end[h:r1] > X))[0]
            S = int(pos[h + open_[0]]) if open_.size else X
            sh["hi_tid"], sh["hi_pos"], sh["next_lo_pos"] = t, X, S
            lo = (t, S, X)
        shards.append(sh)
    return shards, end


def shard_window(sh) -> Window:
    return Window(first=sh["first"], lo_tid=sh["lo_tid"], lo_pos=sh["lo_pos"], cnt_pos=sh["cnt_pos"],
                  hi_tid=sh["hi_tid"], hi_pos=sh["hi_pos"], next_lo_pos=sh["next_lo_pos"])


def shard_final_mask(batch: Batch, sh, end: np.ndarray, done: np.ndarray) -> np.ndarray:
    """which records of [h0, r1) turn final in this shard (not done before, not reaching its right cut)"""
    n = int(batch.n_reads)
    tid = np.ctypeslib.as_array(batch.tid, shape=(n,))
    pos = np.ctypeslib.as_array(batch.pos, shape=(n,))
    idx = np.arange(sh["h0"], sh["r1"])
    fin = ~done[idx]
    if sh["hi_tid"] >= 0:
        in_pileup = end[idx] > pos[idx]
        fin &= ~(in_pileup & (tid[idx] == sh["hi_tid"]) & (end[idx] > sh["hi_pos"]))
    return fin


def run_region_shards(contexts, batch: Batch, n_shards: int):
    """Region shards of one batch on independent contexts (one per GPU, or several on one GPU): every shard starts on its own
    from the reset state, then the saved states are checked in position order and a shard whose incoming state was not
    neutral runs again from the true one.  Returns the merged result and the number of re-runs."""
    shards, end = plan_region_shards(batch, n_shards)
    n = int(batch.n_reads)
    off = np.ctypeslib.as_array(batch.off, shape=(n,))
    subs = [sub_batch(batch, sh["h0"], sh["r1"]) for sh in shards]
    outs = [contexts[k % len(contexts)].process_window(subs[k][0], shard_window(sh)) for k, sh in enumerate(shards)] \
        if len(contexts) >= n_shards else None
    reruns = 0
    if outs is None:                                   # fewer contexts than shards: the sequential chain on one context
        outs = []
        g = contexts[0]
        for k, sh in enumerate(shards):
            w = shard_window(sh)
            if w.first == 2: w.first = 0
            outs.append(g.process_window(subs[k][0], w))
    else:
        spec = [k for k in range(1, n_shards) if shards[k]["first"] == 2]
        in_order = any(contexts[k].carry_is_neutral(contexts[k - 1].carry_export(), shards[k]["lo_tid"], shards[k]["lo_pos"]) < 0 for k in spec)
        for k in spec:
            sh = shards[k]
            carry = contexts[k - 1].carry_export()
            if in_order or contexts[k].carry_is_neutral(carry, sh["lo_tid"], sh["lo_pos"]) != 1:
                contexts[k].carry_import(carry)
                w = shard_window(sh); w.first = 0
                outs[k] = contexts[k].process_window(subs[k][0], w)
                reruns += 1
    qual = np.zeros(int(batch.qual_bytes), dtype=np.uint8)
    done = np.zeros(n, dtype=bool)
    counters = {k: 0 for k in COUNTER_NAMES}
    events = []
    for k, sh in enumerate(shards):
        fin = shard_final_mask(batch, sh, end, done)
        idx = np.arange(sh["h0"], sh["r1"])[fin]
        base = int(off[sh["h0"]])
        oq = outs[k]["qual"]
        if idx.size:
            # one block copy for the long contiguous run, record by record for the ragged edges
            brk = np.nonzero(np.diff(idx) != 1)[0]
            starts = np.concatenate(([0], brk + 1)); stops = np.concatenate((brk + 1, [idx.size]))
            for a, b in zip(starts, stops):
                i0, i1 = int(idx[a]), int(idx[b - 1]) + 1
                q0 = int(off[i0]); q1 = int(off[i1]) if i1 < n else int(batch.qual_bytes)
                qual[q0:q1] = oq[q0 - base: q1 - base]
            done[idx] = True
        for c in COUNTER_NAMES:
            counters[c] += outs[k]["counters"][c]
        events.append(outs[k]["events"])
    assert done.all()
    return {"qual": qual, "events": np.concatenate(events) if events else np.zeros(0, EVENT_DTYPE), "counters": counters,
            "reruns": reruns, "shards": shards}


def algorithmic_bytes(batch: Batch) -> int:
    return int(load_lib().cg_algorithmic_bytes(C.byref(batch)))


def aligned_bases(batch: Batch) -> int:
    return int(load_lib().cg_aligned_bases(C.byref(batch)))


def bed_text(events: np.ndarray, target_names) -> str:
    """BED lines exactly as the reference prints them (snp_score.c:1496-1498 etc.)."""
    return "".join(f"{target_names[e['tid']]}\t{max(int(e['pos']) - 50, 0)}\t{int(e['pos']) + 50}\t{BED_TAGS[e['tag']]}\n"
                   for e in events)


def crumble_cli(argv) -> int:
    """Run the crumble command line (reference main(), snp_score.c:2144) in-process."""
    lib = load_lib()
    args = [b"crumble"] + [a.encode() if isinstance(a, str) else a for a in argv]
    arr = (C.c_char_p * (len(args) + 1))(*args, None)
    return int(lib.crumble_main(len(args), arr))


# ---- synthetic data (libcrumble_sim.so) ------------------------------------------------------
class SimCfg(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("n_contigs", C.c_int), ("contig_len", C.c_int64), ("depth", C.c_double),
                ("read_len", C.c_int), ("qual_binned", C.c_int), ("features_per_mb", C.c_double), ("amplicon", C.c_int),
                ("n_amplicons", C.c_int), ("amplicon_len", C.c_int), ("amplicon_depth", C.c_int),
                ("n_unmapped_tail", C.c_int), ("threads", C.c_int), ("job_first", C.c_int), ("job_count", C.c_int), ("human_like", C.c_int)]


def load_sim():
    global _sim
    if _sim is not None:
        return _sim
    p = LIB_DIR / "libcrumble_sim.so"
    if not p.exists():
        raise CrumbleError(f"{p} is missing (run __graft_entry__.build())")
    s = C.CDLL(str(p))
    s.simgen_preset.argtypes = [C.POINTER(SimCfg), C.c_char_p, C.c_double, C.c_uint64]
    s.simgen_generate.argtypes = [C.POINTER(SimCfg), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t),
                                  C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
    s.simgen_free.argtypes = [C.c_void_p]
    _sim = s
    return s


def simulate(preset: str, scale: float = 1.0, seed: int = 1, threads: int = 0, **cfg_overrides):
    """Synthetic aligned reads (SURVEY.md §8d) as an uncompressed BAM stream (numpy uint8)."""
    s = load_sim()
    cfg = SimCfg()
    if s.simgen_preset(C.byref(cfg), preset.encode(), scale, seed) != 0:
        raise ValueError(f"unknown preset {preset}")
    cfg.threads = threads
    for k, v in cfg_overrides.items():
        setattr(cfg, k, v)
    out = C.c_void_p(); n = C.c_size_t(); nr = C.c_int64(); nb = C.c_int64()
    if s.simgen_generate(C.byref(cfg), C.byref(out), C.byref(n), C.byref(nr), C.byref(nb)) != 0:
        raise CrumbleError("simgen failed")
    arr = np.ctypeslib.as_array(C.cast(out, C.POINTER(C.c_uint8)), shape=(n.value,)).copy()
    s.simgen_free(out)
    return arr, int(nr.value), int(nb.value)
