"""modulate_b200 -- B200-native keystream / archive data-movement path of AdamClixby/Modulate.

The product is ``libmodulate_b200.so`` (hand-written sm_100a kernels behind the C ABI of
``include/modulate_b200.h``) plus the C++ facade classes with the reference's signatures
(``csrc/CEncryptionCycler.h``, ``csrc/CArk.h``).  This Python package is the host-side harness
over that C ABI, mirroring the reference's operator interface for the path:

* ``CEncryptionCycler().Cycle(lpData, liDataSize, liInitialKey)`` -- reference
  ``CEncryptionCycler.h:6``; in place, host or device buffer.
* ``Plan`` / ``cycle_batch`` -- CArk's offset/length table as device descriptors (reference
  ``CArk.cpp:494`` gather, ``:807-811`` scatter) through one variable-length batched kernel.
* ``find_batch`` / ``Plan.find`` / ``ark_find`` -- which entries hold a byte pattern, deciphered and
  matched on the GPU without storing anything; ``PatternSet`` / ``find_set_batch`` / ``Plan.find_set`` /
  ``ark_find_set`` -- the same for up to 256 patterns in one pass; ``mask=`` / ``ignore_case=`` and the helpers
  ``wildcard_pattern`` / ``ignore_case_pattern`` -- wildcard bytes and nibbles, ASCII case folding.
* ``shard_range`` / ``shard_descs`` / ``key_jump`` -- offset-range sharding, one process per GPU;
  ``cycle_sharded`` / ``cycle_batch_sharded`` -- the same split over every GPU inside ONE process.

Nothing here computes keystream on the CPU; every call goes through the CUDA library and raises
``ModError`` if no GPU is usable.
"""
from .api import (ignore_case_pattern, wildcard_pattern, MATCH_DTYPE, SET_MATCH_DTYPE, PatternSet, ark_find, ark_find_set, find_batch, find_set_batch, ArkError, CEncryptionCycler, DESC_DTYPE, ModError, Plan, cycle, cycle_batch, cycle_batch_sharded, group_descs,
                  cycle_device, cycle_sharded, ark_pack, ark_unpack, dta_set_int, device_count, init, key_jump, launch_count, make_descs, shard_descs, shard_range)

__all__ = ["ignore_case_pattern", "wildcard_pattern", "MATCH_DTYPE", "SET_MATCH_DTYPE", "PatternSet", "ark_find", "ark_find_set", "find_batch", "find_set_batch", "ArkError", "ark_pack", "ark_unpack", "dta_set_int", "CEncryptionCycler", "DESC_DTYPE", "ModError", "Plan", "cycle", "cycle_batch", "cycle_batch_sharded", "group_descs", "cycle_device", "cycle_sharded",
           "device_count", "init", "key_jump", "launch_count", "make_descs", "shard_descs", "shard_range"]
