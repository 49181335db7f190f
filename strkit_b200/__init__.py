"""strkit_b200 -- B200-native replacement for STRkit's per-read repeat-count hot path.

Importing this package loads the CUDA shared library (strkit_b200/libstrkit_b200.so); there is no CPU
fallback.  Public surface (mirrors strkit.call.repeats / repeat_count_params / align_matrix):

    get_repeat_count, get_ref_repeat_count      drop-in per-call API
    RepeatCountParams, get_reference_rc_params  search parameters
    Engine, ReadBatch, LocusReads, pack_loci    the batched API (one C-ABI call per block of loci)
    install()                                   rebind the names inside an importable `strkit`
    BlockSession                                block mode: one device call per block of loci, unchanged bookkeeping
    strkit_rust_ext_shim.get_repeat_count       the 9-argument PyO3 signature (repeats.py:58-68)
    call_alleles, call_alleles_batch            bootstrap + GMM allele calls (strkit.call.allele.call_alleles)
    call_alleles_ploidy_batch                   the same with an allele count per locus (1..8)
"""
from .alleles import AlleleCalls, CallData, call_alleles, call_alleles_batch, call_alleles_ploidy_batch
from .batcher import ARENA_ASCII, ARENA_NIBBLE, LocusReads, ReadBatch, pack_loci
from .engine import KERNEL_AUTO, KERNEL_GENERAL, MODE_SG, MODE_SG_QE, DeviceBatch, Engine, default_engine, device_count
from .install import install, uninstall
from .locus_block import BlockSession
from .repeat_count_params import RepeatCountParams, get_reference_rc_params
from .repeats import get_ref_repeat_count, get_repeat_count
from .sharding import count_reads_sharded, partition_catalog

__version__ = "0.1.0"
__all__ = ["LocusReads", "ReadBatch", "pack_loci", "Engine", "DeviceBatch", "default_engine", "device_count",
           "MODE_SG", "MODE_SG_QE", "KERNEL_AUTO", "KERNEL_GENERAL", "RepeatCountParams", "get_reference_rc_params",
           "get_repeat_count", "get_ref_repeat_count", "install", "uninstall", "count_reads_sharded",
           "partition_catalog", "call_alleles", "call_alleles_batch", "call_alleles_ploidy_batch", "AlleleCalls", "CallData", "BlockSession",
           "ARENA_ASCII", "ARENA_NIBBLE"]
