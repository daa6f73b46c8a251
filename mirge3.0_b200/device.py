"""Host-side driver of the CUDA library: contexts, torch-owned device buffers, the collapse table
and the per-batch digest pipeline (tokenise -> line index -> trim -> collapse).

PyTorch is plumbing only here (device memory, streams, the sort used when an index is built);
every byte of the hot path is touched by the kernels in ``csrc/`` through the C ABI."""
from __future__ import annotations

import contextlib
import os
import ctypes as C
from dataclasses import dataclass
from typing import Optional

import numpy as np
import torch

from . import abi
from . import params as P


class MirgeError(RuntimeError):
    pass


class FastqFormatError(MirgeError):
    """Malformed FASTQ input (the reference lets dnaio.FastqFormatError propagate, digest.py:324)."""


class CapacityError(MirgeError):
    pass


def _pow2_at_least(n: int) -> int:
    c = 1
    while c < n:
        c <<= 1
    return c


class Device:
    """One CUDA context of the library bound to ``cuda:<index>`` (one per process / GPU)."""

    def __init__(self, index: int = 0):
        if not torch.cuda.is_available():
            raise MirgeError("mirge_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = abi.load_library()
        self.index = index
        self.tdev = torch.device("cuda", index)
        torch.cuda.set_device(self.tdev)
        ctx = C.c_void_p()
        rc = self.lib.mirge_ctx_create(index, C.byref(ctx))
        if rc != 0:
            raise MirgeError("mirge_ctx_create failed: %s" % self.lib.mirge_last_error(None).decode())
        self.ctx = ctx
        self.trim_params: Optional[abi.TrimParams] = None
        self.slots = 0
        self.launches = 0  # kernels launched through this context (bench.py reports it)
        self.timing = False  # bench.py: CUDA-event timing of the hot kernels on their launch stream
        self._timers = {}

    def __del__(self):
        try:
            if getattr(self, "ctx", None):
                self.lib.mirge_ctx_destroy(self.ctx)
                self.ctx = None
        except Exception:
            pass

    def check(self, rc: int):
        if rc == 0:
            return
        msg = self.lib.mirge_last_error(self.ctx).decode(errors="replace")
        if rc == abi.ERR_FORMAT:
            raise FastqFormatError(msg)
        if rc == abi.ERR_CAPACITY:
            raise CapacityError(msg)
        raise MirgeError("%s (code %d)" % (msg, rc))

    @contextlib.contextmanager
    def timed(self, name: str):
        """Bracket the kernels enqueued inside with CUDA events on the current (launch) stream."""
        if not self.timing:
            yield
            return
        st = torch.cuda.current_stream(self.tdev)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        yield
        b.record(st)
        self._timers.setdefault(name, []).append((a, b))

    def timer_totals(self, reset: bool = True):
        """{name: (n_launch_groups, total_ms)} after synchronising the device."""
        torch.cuda.synchronize(self.tdev)
        out = {k: (len(v), float(sum(a.elapsed_time(b) for a, b in v))) for k, v in self._timers.items()}
        if reset:
            self._timers = {}
        return out

    def stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def set_trim_config(self, cfg: P.TrimConfig):
        p = P.build_trim_params(cfg)
        self.check(self.lib.mirge_set_trim_params(self.ctx, C.byref(p)))
        self.trim_params = p
        self.slots = self.lib.mirge_trim_slots(self.ctx)
        self.cfg = cfg

    def empty(self, n: int, dtype) -> torch.Tensor:
        return torch.empty(max(int(n), 1), dtype=dtype, device=self.tdev)

    def zeros(self, n: int, dtype) -> torch.Tensor:
        return torch.zeros(max(int(n), 1), dtype=dtype, device=self.tdev)


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


class CollapseTable:
    """Torch-owned storage of one ``mirge_table`` plus host mirrors of its counters.  The load factor
    is kept <= 0.5 by ``reserve`` (growth = rehash kernel), so probe sequences stay short."""

    def __init__(self, dev: Device, min_keys: int = 1 << 16, words_per_key: int = 6):
        self.dev = dev
        self.capacity = _pow2_at_least(max(2 * min_keys, 1024))
        self.max_keys = self.capacity // 2
        self.slots = dev.zeros(self.capacity * 4, torch.int32)
        self.arena = dev.empty(self.max_keys * words_per_key, torch.int32)
        self.key_ref = dev.empty(self.max_keys, torch.int32)
        self.ctrl = dev.zeros(8, torch.int64)
        self.n_keys = 0
        self.arena_used = 0
        # share of a batch's insert-list items that created a key (last batch): decides whether the next batch's keys
        # are written straight into the arena (mostly new keys: nothing is copied) or into a batch buffer from which
        # only the new keys are copied (mostly repeats: the arena grows with unique sequences, not with reads)
        self.new_frac = 1.0
        self._struct()

    def _struct(self):
        self.struct = abi.Table(self.slots.data_ptr(), self.capacity, self.arena.data_ptr(), self.arena.numel(),
                                self.key_ref.data_ptr(), self.max_keys, self.ctrl.data_ptr())
        return self.struct

    def reset(self):
        d = self.dev
        d.check(d.lib.mirge_table_reset(d.ctx, C.byref(self.struct), d.stream()))
        self.n_keys = 0
        self.arena_used = 0
        self.new_frac = 1.0

    def check(self):
        """Synchronise, raise on table errors, refresh n_keys / arena_used."""
        d = self.dev
        nk, au = C.c_uint64(0), C.c_uint64(0)
        rc = d.lib.mirge_table_check_sync(d.ctx, C.byref(self.struct), C.byref(nk), C.byref(au), d.stream())
        self.n_keys, self.arena_used = int(nk.value), int(au.value)
        d.check(rc)
        return self.n_keys

    def reserve(self, extra_keys: int, extra_words: int):
        """Make room for ``extra_keys`` new keys / ``extra_words`` arena words (worst case of a batch)."""
        need_keys = self.n_keys + int(extra_keys)
        need_words = self.arena_used + int(extra_words)
        grow_slots = need_keys > self.max_keys
        grow_arena = need_words > self.arena.numel()
        if not grow_slots and not grow_arena:
            return
        d = self.dev
        old = abi.Table(self.slots.data_ptr(), self.capacity, self.arena.data_ptr(), self.arena.numel(),
                        self.key_ref.data_ptr(), self.max_keys, self.ctrl.data_ptr())
        keep = (self.slots, self.arena, self.key_ref)  # keep alive until the rehash has run
        if grow_arena:
            new_arena = d.empty(max(need_words * 3 // 2, 2 * self.arena.numel()), torch.int32)
            new_arena[: self.arena_used].copy_(self.arena[: self.arena_used])
            self.arena = new_arena
        if grow_slots:
            self.capacity = _pow2_at_least(4 * need_keys)
            self.max_keys = self.capacity // 2
            new_ref = d.empty(self.max_keys, torch.int32)
            new_ref[: self.n_keys].copy_(self.key_ref[: self.n_keys])
            self.key_ref = new_ref
            self.slots = d.empty(self.capacity * 4, torch.int32)
            self._struct()
            d.check(d.lib.mirge_table_rehash(d.ctx, C.byref(old), C.byref(self.struct), d.stream()))
            d.launches += 1
        else:
            self._struct()
        torch.cuda.current_stream(d.tdev).synchronize()
        del keep

    def drain(self):
        """(ids int32[n], counts int32[n]) of every key counted since the last drain; zeroes counts."""
        d = self.dev
        self.check()
        n_max = max(self.n_keys, 1)
        ids = d.empty(n_max, torch.int32)
        cnt = d.empty(n_max, torch.int32)
        n_out = d.zeros(1, torch.int64)
        d.check(d.lib.mirge_table_drain(d.ctx, C.byref(self.struct), _ptr(ids), _ptr(cnt), n_max, _ptr(n_out), d.stream()))
        d.launches += 1
        n = int(n_out.item())
        self.check()
        return ids[:n], cnt[:n]

    def _export_device(self, id0: int, n: int):
        """(asc uint8[n * stride] on the device, stride, lens int32[n]): zero-padded ASCII rows of keys [id0, id0 + n)."""
        d = self.dev
        # first pass with a narrow stride to learn the lengths, second pass only if needed
        stride = 64
        while True:
            asc = d.empty(n * stride, torch.uint8)
            lens = d.empty(n, torch.int32)
            d.check(d.lib.mirge_table_export_keys(d.ctx, C.byref(self.struct), id0, n, _ptr(asc), stride, _ptr(lens), d.stream()))
            d.launches += 1
            mx = int(lens.max().item())
            if mx <= stride:
                return asc, stride, lens
            stride = (mx + 15) // 16 * 16

    def export_keys(self, id0: int = 0, n: Optional[int] = None) -> np.ndarray:
        """Keys [id0, id0+n) decoded to a numpy 'S<maxlen>' array (exact original read text)."""
        if n is None:
            n = self.n_keys - id0
        if n <= 0:
            return np.zeros(0, dtype="S1")
        asc, stride, _ = self._export_device(id0, n)
        host = asc.cpu().numpy().reshape(n, stride)
        return np.ascontiguousarray(host).view("S%d" % stride).reshape(n)

    def export_sorted(self, seen: Optional[np.ndarray] = None):
        """(order int64[m], offsets int64[m + 1], data uint8[...]) on the host: the key ids in bytewise order of their text
        (numpy's order for 'S' arrays; only ids with seen[id] when given) and the texts back to back in that order.
        Sorting (LSD radix over big-endian 8-byte chunks of the zero-padded rows), selection and compaction run on
        the device: argsort and slicing of tens of millions of strings on the host take minutes."""
        if self.n_keys <= 0:
            return np.zeros(0, dtype=np.int64), np.zeros(1, dtype=np.int64), np.zeros(0, dtype=np.uint8)
        keep = None if seen is None else torch.from_numpy(np.ascontiguousarray(seen.astype(bool))).to(self.dev.tdev)
        perm, offsets, data = self.export_sorted_device(keep)
        return perm.cpu().numpy(), offsets.cpu().numpy(), data.cpu().numpy()

    def export_sorted_device(self, keep: Optional[torch.Tensor] = None):
        """export_sorted with the three results left on the device (``keep``: bool tensor over the key ids)."""
        d = self.dev
        n = self.n_keys
        if n <= 0:
            z = torch.zeros(0, dtype=torch.int64, device=d.tdev)
            return z, torch.zeros(1, dtype=torch.int64, device=d.tdev), torch.zeros(0, dtype=torch.uint8, device=d.tdev)
        asc, stride, lens = self._export_device(0, n)
        rows = asc.view(n, stride)
        if int((asc >= 128).any().item()):
            # a byte >= 0x80 would flip the sign of its chunk: order on the host (does not happen with FASTQ text)
            keys = np.ascontiguousarray(rows.cpu().numpy()).view("S%d" % stride).reshape(n)
            perm = torch.from_numpy(np.argsort(keys, kind="stable")).to(d.tdev)
        else:
            chunks = rows.view(n, stride // 8, 8).flip(2).contiguous().view(torch.int64).view(n, stride // 8)
            perm = torch.arange(n, device=d.tdev, dtype=torch.int64)
            for c in range(stride // 8 - 1, -1, -1):
                perm = perm[torch.sort(chunks[perm, c], stable=True).indices]
            del chunks
        if keep is not None:
            perm = perm[keep[perm]]
        lens_s = lens[perm].to(torch.int64)
        srt = rows[perm]
        inside = torch.arange(stride, device=d.tdev).unsqueeze(0) < lens_s.unsqueeze(1)
        data = srt[inside]
        offsets = torch.zeros(perm.numel() + 1, dtype=torch.int64, device=d.tdev)
        torch.cumsum(lens_s, 0, out=offsets[1:])
        return perm, offsets, data


@dataclass
class BatchResult:
    n_records: int
    consumed: int
    n_emitted: int
    key_words: int
    line_start: Optional[torch.Tensor] = None
    win: Optional[torch.Tensor] = None
    key_off: Optional[torch.Tensor] = None
    keys: Optional[torch.Tensor] = None
    in_place: bool = False  # keys were written straight into the collapse table's arena
    arena_words: int = 0  # words the batch's keys occupy (repeated slots share a key); key_words counts every emitted key
    ins: Optional[torch.Tensor] = None  # insert list of the collapse: (key word offset, count) of every distinct key a read emitted
    n_items: int = 0


class DigestEngine:
    """tokenise -> trim -> collapse for batches of FASTQ bytes resident on the device."""

    def __init__(self, dev: Device, cfg: P.TrimConfig):
        self.dev = dev
        dev.set_trim_config(cfg)
        self.cfg = cfg
        self.E = dev.slots
        self.trim_mode = 0  # 0 = automatic kernel choice, 1 = always the generic full-DP kernel
        self.INPLACE_MIN_NEW = float(os.environ.get("MIRGE_B200_INPLACE_MIN_NEW", "0.25"))
        dev.check(dev.lib.mirge_trim_mode(dev.ctx, 0))
        self.stats = {"records": 0, "bytes": 0, "emitted": 0, "key_words": 0, "deferred": 0, "dp_reads": 0, "dp_redo": 0}  # running totals (bench.py rooflines)

    def set_trim_mode(self, mode: int):
        self.dev.check(self.dev.lib.mirge_trim_mode(self.dev.ctx, int(mode)))
        self.trim_mode = int(mode)

    def trim_batch(self, buf: torch.Tensor, nbytes: int, is_final: bool, keep: bool = True,
                   table: Optional["CollapseTable"] = None) -> BatchResult:
        """tokenise -> line index -> trim of buf[:nbytes] (uint8, device), with every kernel choice of mirge_trim (split
        bit-parallel pipeline, generic full DP, qiagen UMIs).  Returns the device arrays the collapse consumes (and the
        parity tests read).  With ``table`` the packed keys are written straight into that table's arena (zero-copy
        collapse); otherwise into a batch buffer."""
        if nbytes == 0:
            return BatchResult(0, 0, 0, 0)
        d, lib, E = self.dev, self.dev.lib, self.E
        st = d.stream()
        scratch = d.empty(lib.mirge_tokenise_scratch_bytes(nbytes), torch.uint8)
        n_rec, consumed = C.c_uint64(0), C.c_uint64(0)
        with d.timed("tokenise"):
            d.check(lib.mirge_tokenise_sync(d.ctx, _ptr(buf), nbytes, 1 if is_final else 0, _ptr(scratch),
                                            C.byref(n_rec), C.byref(consumed), st))
        d.launches += 3 if not is_final else 2
        n = int(n_rec.value)
        if n == 0:
            return BatchResult(0, int(consumed.value), 0, 0)
        used = int(consumed.value)
        line_start = d.empty(4 * n + 4, torch.int32)
        # same nbytes as the census: the scratch layout depends on it
        with d.timed("line_index"):
            d.check(lib.mirge_line_index(d.ctx, _ptr(buf), nbytes, _ptr(scratch), _ptr(line_start), n, st))
        d.launches += 3
        # per-slot windows / key offsets are what the parity tests read; the product path (keep=False) only wants the
        # insert list of the collapse
        win = d.empty(n * E * 4, torch.int16) if keep else None
        key_off = d.empty(n * E, torch.int32) if keep else None
        ins = d.empty(n * E, torch.int64)
        slow = d.empty(lib.mirge_trim_scratch_bytes(n), torch.uint8)  # work lists of the split trim pipeline
        cap = E * (2 * n + used // 24) + 4096
        mode = self.trim_mode
        base_words = 0
        if table is not None and table.new_frac < self.INPLACE_MIN_NEW:
            table = None  # repeats dominate: batch key buffer + copying insert keeps the arena tight
        if table is not None:
            table.check()
            base_words = table.arena_used
        for attempt in range(4):
            ctrl = d.zeros(16, torch.int64)
            if table is not None:
                table.reserve(0, cap)  # room in the arena for this batch's keys
                keys = table.arena
                ctrl[0:1].fill_(base_words)
                cap_abs = int(table.arena.numel())
            else:
                keys = d.empty(cap, torch.int32)
                cap_abs = cap
            if mode != self.trim_mode:
                d.check(lib.mirge_trim_mode(d.ctx, mode))
            try:
                with d.timed("trim"):
                    d.check(lib.mirge_trim(d.ctx, _ptr(buf), used, _ptr(line_start), n, _ptr(win), _ptr(key_off),
                                           _ptr(keys), cap_abs, _ptr(ctrl), _ptr(slow), _ptr(ins), n * E, st))
            finally:
                if mode != self.trim_mode:
                    d.check(lib.mirge_trim_mode(d.ctx, self.trim_mode))
            d.launches += 4
            c = ctrl.cpu().numpy().view(np.uint64)
            # ctrl[0] = insert-list entries << 36 | key words (one atomic hands out both, csrc/trim.cu)
            words_used, n_items = int(c[0]) & ((1 << 36) - 1), int(c[0]) >> 36
            flags = int(c[2])
            self.stats["deferred"] += int(c[5])  # reads handed to the whole-pipeline second pass (diagnostics)
            self.stats["dp_reads"] += int(c[6])  # reads whose adapter search ran the bit-vector DP
            self.stats["dp_redo"] += int(c[7])  # of those, searches that needed cost columns
            if flags & 8 and mode != 1:
                # a record group did not fit the bit-parallel kernel's shared-memory staging:
                # repeat the batch with the generic kernel (same results, slower)
                mode = 1
                continue
            if flags & 1:
                rec = int(np.uint64(~c[3]))
                raise FastqFormatError("FASTQ format error in record %d of the batch (header must start with '@', "
                                       "line 3 with '+', sequence and qualities must have equal length)" % rec)
            if flags & 4:
                raise MirgeError("read longer than %d bases is not supported" % abi.MAX_READ_LEN)
            if flags & 2:
                if attempt >= 2:
                    raise CapacityError("trim: key buffer overflow")
                cap = E * (n + used // 2 + used // 32 + 64) + 4096  # worst case: every base an exception
                continue
            break
        if table is not None:
            table.arena_used = words_used
            table.ctrl[0:1].fill_(table.arena_used)  # the table's own counter of arena words in use
            return BatchResult(n, used, int(c[1]), int(c[4]), line_start if keep else None, win, key_off, None, True,
                               words_used - base_words, ins, n_items)
        return BatchResult(n, used, int(c[1]), int(c[4]), line_start if keep else None, win, key_off, keys, False,
                           words_used, ins, n_items)

    def collapse_batch(self, table: CollapseTable, br: BatchResult):
        """completeDict[key] += 1 for every key the trim kernel emitted."""
        st_ = self.stats
        st_["records"] += br.n_records
        st_["bytes"] += br.consumed
        st_["emitted"] += br.n_emitted
        st_["key_words"] += br.key_words
        if br.n_records == 0 or br.n_emitted == 0:
            return
        d, lib = self.dev, self.dev.lib
        scratch = d.empty(2 * br.n_items, torch.int32)
        if br.in_place:
            table.reserve(br.n_items, 0)
            keys = table.arena
        else:
            table.check()
            table.reserve(br.n_items, br.arena_words)
            keys = br.keys
        with d.timed("collapse"):
            d.check(lib.mirge_collapse_insert_list(d.ctx, C.byref(table.struct), _ptr(keys), _ptr(br.ins), br.n_items,
                                                   _ptr(scratch), d.stream()))
        d.launches += 4
        before = table.n_keys
        table.check()
        table.new_frac = (table.n_keys - before) / max(br.n_items, 1)

    def digest_device(self, buf: torch.Tensor, table: CollapseTable, batch_bytes: int = 256 << 20, on_piece=None) -> int:
        """Whole sample resident on the device: returns the number of records parsed.  ``on_piece(table)`` runs
        after every collapsed batch (streamed annotation of the keys it created)."""
        total = int(buf.numel())
        pos = 0
        n_records = 0
        while pos < total:
            end = min(total, pos + batch_bytes)
            final = end == total
            view = buf[pos:end]
            br = self.trim_batch(view, end - pos, final, keep=False, table=table)
            if br.n_records == 0 and not final:
                if end - pos >= batch_bytes and batch_bytes >= (1 << 20):
                    raise FastqFormatError("FASTQ record does not fit into a batch")
            self.collapse_batch(table, br)
            if on_piece is not None:
                on_piece(table)
            n_records += br.n_records
            if br.consumed == 0 and not final:
                raise FastqFormatError("no complete FASTQ record in batch")
            pos += br.consumed if not final else (end - pos)
        return n_records

    @staticmethod
    def max_batches(total_bytes: int, batch_bytes: int, max_record: int = 1 << 16) -> int:
        """Upper bound of the batches digest_device* cuts ``total_bytes`` into (a batch ends at a record boundary)."""
        step = max(batch_bytes - max_record, 1)
        return (int(total_bytes) + step - 1) // step

    def digest_device_exchange(self, buf: torch.Tensor, locals2, worker, batch_bytes: int = 256 << 20, n_batches: int = 0) -> int:
        """Multi-GPU form of digest_device (one process per GPU): every batch is collapsed into one of two local tables
        and its (key, count) pairs are handed to ``worker`` (distributed.ExchangeWorker), which partitions them by
        owner, runs the all-to-all and merges into the owner table on its own stream while the next batch is trimmed
        here into the other local table.  Collective: every rank must submit the same number of exchanges -- pass
        ``n_batches`` = the maximum over the ranks of ``max_batches(...)`` and a rank that runs out of input keeps
        submitting empty exchanges."""
        total = int(buf.numel())
        pos, k, n_records = 0, 0, 0
        handles = [None, None]
        for t in locals2:
            t.reset()
        while pos < total:
            tab = locals2[k % 2]
            if handles[k % 2] is not None:
                handles[k % 2].wait()  # the exchange that read this table is done
                tab.reset()
            end = min(total, pos + batch_bytes)
            final = end == total
            br = self.trim_batch(buf[pos:end], end - pos, final, keep=False, table=tab)
            self.collapse_batch(tab, br)
            with self.dev.timed("drain"):
                ids, cnt = tab.drain()
            handles[k % 2] = worker.submit(tab, ids, cnt)
            n_records += br.n_records
            if br.consumed == 0 and not final:
                raise FastqFormatError("no complete FASTQ record in batch")
            pos += br.consumed if not final else (end - pos)
            k += 1
        empty = torch.zeros(0, dtype=torch.int32, device=self.dev.tdev)
        while k < n_batches:  # keep the collectives of all ranks in step
            worker.submit(locals2[0], empty, empty)
            k += 1
        return n_records

