"""Engine: one native context (one GPU) + the calls the batcher makes across the C ABI."""
from __future__ import annotations

import collections
import ctypes as C
import os
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import Iterable, Iterator

import numpy as np

from . import _native
from ._native import check, lib
from .align_matrix import dna_matrix, indel_penalty
from .batcher import ReadBatch
from .repeat_count_params import RepeatCountParams

__all__ = ["Engine", "DeviceBatch", "default_engine", "MODE_SG", "MODE_SG_QE", "KERNEL_AUTO", "KERNEL_GENERAL"]

MODE_SG = 15      # parasail "sg": all four ends free (the mode the read path is believed to use)
MODE_SG_QE = 2    # parasail "sg_qe" (repeats.py:33,40)
KERNEL_AUTO = 0
KERNEL_GENERAL = 1
STAT_NAMES = ("executed_cells", "reference_cells", "kernel_launches", "dp_ms", "replay_ms", "widening_passes",
              "reads_packed_kernel", "reads_general_kernel")


def _p(a: np.ndarray) -> int:
    return a.ctypes.data


def _ascii_only(batch: ReadBatch) -> None:
    if batch.arena_format != 0:
        raise ValueError("this entry point takes ASCII arenas (the nibble format is for the read-path batches)")


class DeviceBatch:
    """A ReadBatch resident in HBM (strk_batch_upload)."""

    def __init__(self, engine: "Engine", handle: int, n_reads: int, n_loci: int):
        self.engine, self.handle, self.n_reads, self.n_loci = engine, handle, n_reads, n_loci

    def free(self) -> None:
        if self.handle:
            lib.strk_batch_free(self.engine._ctx, self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Engine:
    def __init__(self, device: int = 0, end_flags: int = MODE_SG, tie_flags: int = 0,
                 matrix: np.ndarray = dna_matrix, gap_open: int = indel_penalty, gap_extend: int = indel_penalty):
        mat = np.ascontiguousarray(matrix, dtype=np.int8)
        if mat.shape != (17, 17):
            raise ValueError("matrix must be 17x17")
        ctx = C.c_void_p()
        check(lib.strk_init(device, _p(mat), gap_open, gap_extend, end_flags, tie_flags, C.byref(ctx)))
        self._ctx = ctx
        self.device = device
        self.end_flags = end_flags
        self._init_args = (device, end_flags, tie_flags, mat, gap_open, gap_extend)
        self._twin: "Engine | None" = None       # second native context on the same GPU (count_reads_stream)
        self._stream_batch = None                # reusable strk_batch of this context
        self._run_lock = threading.Lock()
        # native contexts are not re-entrant: the per-call drop-in wrappers (which the reference may call from a
        # multiprocessing.dummy thread pool) hold this lock around their C-ABI calls
        self.lock = threading.RLock()
        self.launches = 0    # kernels launched by the streamed path of this context (count_reads_stream accumulates it)

    @property
    def total_launches(self) -> int:
        """Kernels launched by count_reads_stream on this GPU so far (both contexts)."""
        return (self.launches + (self._twin.launches if self._twin else 0) +
                sum(e.launches for e in (getattr(self, "_ref_engs", None) or [])))

    def sync(self) -> None:
        """Wait for everything queued on the context's streams (strk_sync)."""
        check(lib.strk_sync(self._ctx))
        if getattr(self, "_twin", None):
            self._twin.sync()

    def close(self) -> None:
        if getattr(self, "_aux_pool", None):
            self._aux_pool.shutdown(wait=True)
            self._aux_pool = None
        for e in getattr(self, "_ref_engs", None) or []:
            e.close()
        self._ref_engs = None
        if getattr(self, "_twin", None):
            self._twin.close()
            self._twin = None
        if getattr(self, "_ctx", None):
            if self._stream_batch:
                lib.strk_batch_free(self._ctx, self._stream_batch)
                self._stream_batch = None
            lib.strk_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ read path
    def upload(self, batch: ReadBatch) -> DeviceBatch:
        batch.validate()
        h = C.c_void_p()
        check(lib.strk_batch_create(self._ctx, C.byref(h)))
        try:
            check(lib.strk_batch_fill_fmt(self._ctx, h, batch.arena_format, _p(batch.arena), batch.arena.nbytes,
                                          _p(batch.seq_off), _p(batch.lens), _p(batch.est_cn), batch.n_reads,
                                          _p(batch.read_begin), _p(batch.motif_off), _p(batch.motif_len), batch.n_loci))
        except Exception:
            lib.strk_batch_free(self._ctx, h)
            raise
        return DeviceBatch(self, h, batch.n_reads, batch.n_loci)

    def run(self, dbatch: DeviceBatch, rc_params: RepeatCountParams, kernel: int = KERNEL_AUTO, stream: int = 0) -> None:
        check(lib.strk_batch_run(self._ctx, dbatch.handle, rc_params.max_iters, rc_params.initial_local_search_range,
                                 rc_params.initial_step_size, kernel, C.c_void_p(stream)))

    def download(self, dbatch: DeviceBatch, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty((dbatch.n_reads, 4), dtype=np.int32)
        check(lib.strk_batch_download(self._ctx, dbatch.handle, _p(out)))
        return out

    def count_reads(self, batch: ReadBatch, rc_params: RepeatCountParams, kernel: int = KERNEL_AUTO,
                    out: np.ndarray | None = None) -> np.ndarray:
        """out[r] = (best_n, best_score, n_explored, start_count used); host buffers in, host buffer out."""
        batch.validate()
        if out is None:
            out = np.empty((batch.n_reads, 4), dtype=np.int32)
        check(lib.strk_count_reads_fmt(self._ctx, batch.arena_format, _p(batch.arena), batch.arena.nbytes,
                                       _p(batch.seq_off), _p(batch.lens), _p(batch.est_cn), batch.n_reads,
                                       _p(batch.read_begin), _p(batch.motif_off), _p(batch.motif_len), batch.n_loci,
                                       rc_params.max_iters, rc_params.initial_local_search_range,
                                       rc_params.initial_step_size, kernel, _p(out)))
        return out

    def _stream_step(self, batch: ReadBatch, rc_params: RepeatCountParams, kernel: int, out: np.ndarray,
                     run_lock: threading.Lock, ref=None):
        """fill (H2D + device-side planning) -> run (kernels) -> download (D2H) on this context's reusable batch.
        Only the run phase holds `run_lock`: the copies of one block overlap the kernels of the other context.
        ref = (ref_batch, start_count, ref_size, rc[n, 3], vcf_anchor_size, out[n, 8]): the block's reference windows
        (get_ref_repeat_count, once per locus) go through strk_ref_counts between the fill and the run phase."""
        if self._stream_batch is None:
            h = C.c_void_p()
            check(lib.strk_batch_create(self._ctx, C.byref(h)))
            self._stream_batch = h
        check(lib.strk_batch_fill_fmt(self._ctx, self._stream_batch, batch.arena_format, _p(batch.arena),
                                      batch.arena.nbytes, _p(batch.seq_off), _p(batch.lens), _p(batch.est_cn), batch.n_reads,
                                      _p(batch.read_begin), _p(batch.motif_off), _p(batch.motif_len), batch.n_loci))
        if ref is not None:
            # Outside the run lock on purpose: the reference windows of block i + 1 (many small launches, a tenth of the
            # block's cells) run while the other context is in the read kernels of block i and fill the slots those
            # leave idle at the tails of their launches.  (Measured against the alternatives: inside the lock 50.4 M
            # reads x loci/s, here ~60 M, on a third context from a thread of its own 56.2 M, on two of those 57.8 M --
            # under the persistent read CTAs a reference block is latency-bound, and this thread has the slack.)
            rb, start, ref_size, rc, anchor, ref_out = ref
            check(lib.strk_ref_counts(self._ctx, _p(rb.arena), rb.arena.nbytes, _p(rb.seq_off), _p(rb.lens), _p(start),
                                      _p(ref_size), _p(rc), rb.n_loci, _p(rb.motif_off), _p(rb.motif_len), anchor, 0,
                                      _p(ref_out)))
            self.launches += int(self.stats()["kernel_launches"])
        with run_lock:
            check(lib.strk_batch_run(self._ctx, self._stream_batch, rc_params.max_iters,
                                     rc_params.initial_local_search_range, rc_params.initial_step_size, kernel, None))
            self.launches += int(self.stats()["kernel_launches"])
        check(lib.strk_batch_download(self._ctx, self._stream_batch, _p(out)))
        return out if ref is None else (out, ref[5])

    def count_reads_stream(self, batches: Iterable[ReadBatch], rc_params: RepeatCountParams, kernel: int = KERNEL_AUTO,
                           outs: Iterable[np.ndarray] | None = None, refs: Iterable[tuple] | None = None) -> Iterator:
        """count_reads over a stream of locus blocks (the reference's worker pool consumes the catalog block by
        block, call_sample.py:413-420), results yielded in block order.  Two native contexts on this GPU take
        alternate blocks from two host threads: block i+1 is copied to the device and planned while block i is
        in the DP kernels, so the PCIe copy disappears behind the compute.  Pin the host arrays
        (strk_host_register / torch pinned memory) or the copies cannot overlap.
        refs: per block (ref_batch, start_count int32[n], ref_size int32[n], rc int32[n, 3], vcf_anchor_size,
        out int32[n, 8]) -- the reference windows of the block's loci (get_ref_repeat_count, call_locus.py:799-810);
        the stream then yields (reads_out, ref_out) per block: the whole hot path of a block of loci."""
        if self._twin is None:
            d, ef, tf, mat, go, ge = self._init_args
            self._twin = Engine(d, ef, tf, mat, go, ge)
        slots = (self, self._twin)
        out_it = iter(outs) if outs is not None else None
        ref_it = iter(refs) if refs is not None else None
        pending: collections.deque = collections.deque()
        with ThreadPoolExecutor(max_workers=2, thread_name_prefix="strk-stream") as pool:
            for i, batch in enumerate(batches):
                if len(pending) == 2:  # the slot of block i is free once block i-2 is done
                    yield pending.popleft().result()
                batch.validate()
                out = next(out_it) if out_it is not None else np.empty((batch.n_reads, 4), dtype=np.int32)
                ref = next(ref_it) if ref_it is not None else None
                pending.append(pool.submit(slots[i % 2]._stream_step, batch, rc_params, kernel, out, self._run_lock, ref))
            while pending:
                yield pending.popleft().result()

    # ------------------------------------------------------------------ raw tables
    def score_tables(self, batch: ReadBatch, n_lo: np.ndarray, n_hi: np.ndarray, kernel: int = KERNEL_AUTO):
        """Scores of every candidate size in [n_lo[r], n_hi[r]] for every read; returns (scores, out_off)."""
        batch.validate()
        _ascii_only(batch)
        n_lo = np.ascontiguousarray(n_lo, dtype=np.int32)
        n_hi = np.ascontiguousarray(n_hi, dtype=np.int32)
        width = (n_hi.astype(np.int64) - n_lo + 1)
        out_off = np.zeros(batch.n_reads, dtype=np.uint64)
        out_off[1:] = np.cumsum(width)[:-1]
        scores = np.empty(int(width.sum()), dtype=np.int32)
        motif_idx = np.repeat(np.arange(batch.n_loci, dtype=np.int32), np.diff(batch.read_begin)).astype(np.int32)
        check(lib.strk_score_tables(self._ctx, _p(batch.arena), batch.arena.nbytes, _p(batch.seq_off), _p(batch.lens),
                                    _p(motif_idx), _p(n_lo), _p(n_hi), batch.n_reads, _p(batch.motif_off),
                                    _p(batch.motif_len), batch.n_loci, _p(out_off), kernel, _p(scores)))
        return scores, out_off

    def ref_boundary_tables(self, batch: ReadBatch, n_lo: np.ndarray, n_hi: np.ndarray, kernel: int = KERNEL_AUTO):
        """score_ref_boundaries for a window of sizes; one 'read' (the reference window) per locus.
        Returns (table[k] = (fwd_score, fwd_end_query, rev_score, rev_end_query), out_off)."""
        batch.validate()
        _ascii_only(batch)
        if batch.n_reads != batch.n_loci:
            raise ValueError("reference batches hold exactly one sequence per locus")
        n_lo = np.ascontiguousarray(n_lo, dtype=np.int32)
        n_hi = np.ascontiguousarray(n_hi, dtype=np.int32)
        width = (n_hi.astype(np.int64) - n_lo + 1)
        out_off = np.zeros(batch.n_loci, dtype=np.uint64)
        out_off[1:] = np.cumsum(width)[:-1]
        out = np.empty((int(width.sum()), 4), dtype=np.int32)
        check(lib.strk_ref_boundary_tables(self._ctx, _p(batch.arena), batch.arena.nbytes, _p(batch.seq_off),
                                           _p(batch.lens), _p(n_lo), _p(n_hi), batch.n_loci, _p(batch.motif_off),
                                           _p(batch.motif_len), _p(out_off), kernel, _p(out)))
        return out, out_off

    def ref_counts(self, batch: ReadBatch, start_count, ref_size, rc_params, vcf_anchor_size: int,
                   respect_coords: bool = False, out: np.ndarray | None = None) -> np.ndarray:
        """get_ref_repeat_count for every locus of a reference batch; rc_params int32 [n_loci, 3]."""
        batch.validate()
        _ascii_only(batch)
        start_count = np.ascontiguousarray(start_count, dtype=np.int32)
        ref_size = np.ascontiguousarray(ref_size, dtype=np.int32)
        rc = np.ascontiguousarray(rc_params, dtype=np.int32).reshape(batch.n_loci, 3)
        if out is None:
            out = np.empty((batch.n_loci, 8), dtype=np.int32)
        check(lib.strk_ref_counts(self._ctx, _p(batch.arena), batch.arena.nbytes, _p(batch.seq_off), _p(batch.lens),
                                  _p(start_count), _p(ref_size), _p(rc), batch.n_loci, _p(batch.motif_off),
                                  _p(batch.motif_len), vcf_anchor_size, int(respect_coords), _p(out)))
        return out

    def ref_counts_async(self, batch: ReadBatch, start_count, ref_size, rc_params, vcf_anchor_size: int,
                         respect_coords: bool = False, out_buf: np.ndarray | None = None):
        """ref_counts on a native context of its own, from a helper thread: returns a Future of (out, stats).
        A block's reference windows (a tenth of its cells, many small launches) then run UNDER the read kernels the
        caller launches meanwhile on this context (Engine.run / count_reads) instead of before them."""
        if getattr(self, "_ref_engs", None) is None:
            d, ef, tf, mat, go, ge = self._init_args
            self._ref_engs = [Engine(d, ef, tf, mat, go, ge)]   # a context of its own (the streamed path keeps two for reads)
            self._aux_pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="strk-ref")
        ref_eng = self._ref_engs[0]

        def job():
            with ref_eng.lock:
                out = ref_eng.ref_counts(batch, start_count, ref_size, rc_params, vcf_anchor_size, respect_coords, out=out_buf)
                st = ref_eng.stats()
                ref_eng.launches += int(st["kernel_launches"])
            return out, st

        return self._aux_pool.submit(job)

    def measure_int_peak(self) -> dict[str, float]:
        """Measured integer issue rates (1e12 lane-instructions/s): the DP kernels' roofline denominator."""
        s = np.zeros(3, dtype=np.float64)
        check(lib.strk_measure_int_peak(self._ctx, _p(s)))
        return {"alu_pipe": float(s[0]), "fma_pipe": float(s[1]), "dual_pipe": float(s[2])}

    def stats(self) -> dict[str, float]:
        s = np.zeros(8, dtype=np.float64)
        check(lib.strk_get_stats(self._ctx, _p(s)))
        return dict(zip(STAT_NAMES, s.tolist()))


_default: dict[tuple[int, int, int], Engine] = {}
_default_lock = threading.Lock()


def _forget_engines_after_fork() -> None:
    # A CUDA context does not survive fork(): a child (the reference's NonDaemonicPool workers) must build its own
    # engine.  The parent's handles are dropped without being destroyed -- they are not valid in this process.
    for eng in _default.values():
        eng._ctx = None
        eng._twin = None
        eng._stream_batch = None
    _default.clear()


if hasattr(os, "register_at_fork"):
    os.register_at_fork(after_in_child=_forget_engines_after_fork)


def default_engine(device: int = 0, end_flags: int = MODE_SG, tie_flags: int = 0) -> Engine:
    """Per-process engine used by the drop-in get_repeat_count / get_ref_repeat_count wrappers."""
    key = (device, end_flags, tie_flags)
    with _default_lock:
        eng = _default.get(key)
        if eng is None:
            eng = _default[key] = Engine(device, end_flags, tie_flags)
        return eng


def device_count() -> int:
    return int(lib.strk_device_count())


_ = _native  # keep the loader import explicit: importing this module requires the native library
