"""crumble_b200 — B200-native consensus + quality-rewrite hot path of Crumble.

The product is the C-ABI shared library ``lib/libcrumble_gpu.so`` (hand-written sm_100a
kernels, see ``csrc/``); this package is the thin Python mirror used by the tests and
``bench.py``.  See DESIGN.md.
"""
from .api import (  # noqa: F401
    BatchBuilder, Crumble, MultiCrumble, CrumbleError, Params, Window, default_params, simulate, algorithmic_bytes,
    aligned_bases, bed_text, batch_ends, sub_batch, plan_region_shards, run_region_shards, shard_window, shard_final_mask, crumble_cli, load_lib, lib_path, device_batch, concat_fields, DevBatch, COUNTER_NAMES, BED_TAGS, EXPORTS,
    DeviceStream, StreamOut, split_device_batch,
)
