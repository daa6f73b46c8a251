"""``bwtAlign`` -- drop-in for mirge/libs/manifoldAlign.py:68 (same signature, same DataFrame and
run.log side effects) that runs the ordered annotation rounds on the GPU instead of spawning
bowtie ten times and parsing SAM text (manifoldAlign.py:12-64)."""
from __future__ import annotations

import ctypes as C
import os
import time
from pathlib import Path
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import abi
from .device import CollapseTable, Device, MirgeError, _ptr
from .libraries import ROUND_LIBS, LibrarySet, round_policies

_DEVICE: Optional[Device] = None
_LIB_CACHE: Dict[Tuple, LibrarySet] = {}


def get_device(index: int = 0) -> Device:
    """Process-wide context (one per GPU process)."""
    global _DEVICE
    if _DEVICE is None or _DEVICE.index != index:
        _DEVICE = Device(index)
    return _DEVICE


class KeySet:
    """Unique sequences resident on the device in packed-key form, id = row index."""

    def __init__(self, dev: Device, arena: torch.Tensor, key_ref: torch.Tensor, n: int):
        self.dev, self.arena, self.key_ref, self.n = dev, arena, key_ref, n
        self._dummy_slots = dev.zeros(8, torch.int32)
        self._ctrl = dev.zeros(8, torch.int64)
        self.struct = abi.Table(self._dummy_slots.data_ptr(), 2, arena.data_ptr(), arena.numel(), key_ref.data_ptr(),
                                max(n, 1), self._ctrl.data_ptr())

    @classmethod
    def from_table(cls, table: CollapseTable) -> "KeySet":
        table.check()
        return cls(table.dev, table.arena, table.key_ref, table.n_keys)

    @classmethod
    def from_strings(cls, dev: Device, seqs: Sequence) -> "KeySet":
        """Pack Python strings / bytes (the DataFrame index) with the mirge_pack_keys kernel."""
        n = len(seqs)
        if n == 0:
            return cls(dev, dev.zeros(1, torch.int32), dev.zeros(1, torch.int32), 0)
        if isinstance(seqs, np.ndarray) and seqs.dtype.kind == "S":
            lens = np.char.str_len(seqs).astype(np.int64)
            blob = b"".join(seqs.tolist())
        else:
            enc = [s.encode("latin-1") if isinstance(s, str) else bytes(s) for s in seqs]
            lens = np.fromiter((len(b) for b in enc), dtype=np.int64, count=n)
            blob = b"".join(enc)
        if len(lens) and int(lens.max()) > abi.MAX_READ_LEN:
            raise MirgeError("sequence longer than %d bases" % abi.MAX_READ_LEN)
        off = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lens, out=off[1:])
        d_ascii = torch.frombuffer(bytearray(blob) if blob else bytearray(1), dtype=torch.uint8).to(dev.tdev)
        d_off = torch.from_numpy(off).to(dev.tdev)
        words = dev.empty(n, torch.int32)
        dev.check(dev.lib.mirge_key_sizes(dev.ctx, _ptr(d_ascii), _ptr(d_off), n, _ptr(words), dev.stream()))
        csum = torch.cumsum(words.to(torch.int64), 0)
        total = int(csum[-1].item())
        if total >= (1 << 32) - 16:
            raise MirgeError("too many sequences for one key set")
        key_off64 = csum - words.to(torch.int64)
        key_off = torch.where(key_off64 >= (1 << 31), key_off64 - (1 << 32), key_off64).to(torch.int32)
        arena = dev.empty(total, torch.int32)
        dev.check(dev.lib.mirge_pack_keys(dev.ctx, _ptr(d_ascii), _ptr(d_off), n, _ptr(key_off), _ptr(arena), dev.stream()))
        dev.launches += 2
        return cls(dev, arena, key_off, n)


def annotate_keys(dev: Device, libs: LibrarySet, keys: KeySet, spike_in: bool = False, fused: bool = True, split: bool = True,
                  out=None):
    """Run rounds 0..8 (0..9 with spike-ins) in miRge's order (manifoldAlign.py:86-135).
    Returns device tensors (annot_round uint8[n] with 0xFF = unannotated, hit int64[n]).
    ``split`` (default): a streaming pass leaves a round mask per sequence (seed-piece filters of all rounds), then
    warps compact and search their sequences round by round; ``fused`` without ``split``: one thread per sequence
    runs all rounds; neither: one whole-table launch per round."""
    n = keys.n
    if out is not None:  # caller-provided result arrays (initialised to 0xFF / -1 by the caller)
        annot, hit = out
    else:
        annot = torch.full((max(n, 1),), 0xFF, dtype=torch.uint8, device=dev.tdev)
        hit = torch.full((max(n, 1),), -1, dtype=torch.int64, device=dev.tdev)
    if n == 0:
        return annot[:0], hit[:0]
    pols = round_policies()
    n_rounds = 10 if spike_in else 9
    if fused:
        # all rounds in one launch: every key is read once and leaves at the first round that hits it
        lib_arr = (abi.Library * n_rounds)(*[libs[ROUND_LIBS[r]].struct for r in range(n_rounds)])
        pol_arr = (abi.RoundPolicy * n_rounds)(*pols[:n_rounds])
        scratch = dev.empty(dev.lib.mirge_annotate_scratch_bytes(n) // 8 + 1, torch.int64) if split else None
        with dev.timed("annotate"):
            dev.check(dev.lib.mirge_annotate_rounds(dev.ctx, lib_arr, pol_arr, n_rounds, C.byref(keys.struct), n,
                                                    _ptr(annot), _ptr(hit), _ptr(scratch), dev.stream()))
        dev.launches += 3 if split else 1
        return annot[:n], hit[:n]
    for rnd in range(n_rounds):
        lib = libs[ROUND_LIBS[rnd]]
        with dev.timed("annotate_r%d" % rnd):
            dev.check(dev.lib.mirge_annotate_round(dev.ctx, C.byref(lib.struct), C.byref(pols[rnd]), C.byref(keys.struct), n,
                                                   _ptr(annot), _ptr(hit), dev.stream()))
        dev.launches += 1
    return annot[:n], hit[:n]


class StreamedAnnotator:
    """Per-piece hook (``HostStreamer.run(on_piece=...)`` / ``DigestEngine.digest_device(on_piece=...)``) for
    single-GPU runs: after every collapsed piece the keys that piece created are annotated -- a key's annotation
    depends on nothing but its text -- on a side stream, so the (latency-bound) annotation kernel shares the SMs
    with the (issue-bound) trim kernels of the next piece.  With ``to_host`` the new arena words, key offsets,
    annotation rounds and hit words are also copied to pinned host buffers on a third stream, so the D2H of the
    result table overlaps the H2D of the following pieces; only the per-sample counts are left for the end."""

    def __init__(self, dev: Device, libs: LibrarySet, spike_in: bool = False, to_host: bool = True):
        self.dev, self.libs, self.spike, self.copy_out = dev, libs, spike_in, to_host
        self.ann = torch.cuda.Stream(device=dev.tdev)
        self.d2h = torch.cuda.Stream(device=dev.tdev)
        self.host: Dict[str, torch.Tensor] = {}
        self.annot_d: Optional[torch.Tensor] = None  # annotation round / hit word of every key id, on the device
        self.hit_d: Optional[torch.Tensor] = None
        self.reset()

    def reset(self):
        self.n_done = 0
        self.w_done = 0
        self.d2h_bytes = 0

    def _host(self, name: str, dtype, need: int, used: int) -> torch.Tensor:
        buf = self.host.get(name)
        if buf is None or buf.numel() < need:
            new = torch.empty(max(int(need * 1.5), 1 << 20), dtype=dtype).pin_memory()
            if buf is not None and used:
                self.d2h.synchronize()
                new[:used].copy_(buf[:used])
            self.host[name] = buf = new
        return buf

    def to_host(self, name: str, src: torch.Tensor, at: int, used: int):
        """src -> host[name][at : at + len(src)] on the D2H stream (after the work queued on the main stream)."""
        n = int(src.numel())
        if n == 0:
            return
        dst = self._host(name, src.dtype, at + n, used)
        src.record_stream(self.d2h)
        dst[at : at + n].copy_(src, non_blocking=True)
        self.d2h_bytes += n * src.element_size()

    def _device_results(self, need: int):
        """annot_d / hit_d with room for ``need`` keys (grown on the annotation stream, contents kept)."""
        if self.annot_d is None or self.annot_d.numel() < need:
            cap = max(int(need * 1.5), 1 << 20)
            with torch.cuda.stream(self.ann):
                a = torch.empty(cap, dtype=torch.uint8, device=self.dev.tdev)
                h = torch.empty(cap, dtype=torch.int64, device=self.dev.tdev)
                if self.annot_d is not None and self.n_done:
                    a[: self.n_done].copy_(self.annot_d[: self.n_done])
                    h[: self.n_done].copy_(self.hit_d[: self.n_done])
            self.annot_d, self.hit_d = a, h

    def __call__(self, table: CollapseTable):
        n0, w0, n1, w1 = self.n_done, self.w_done, table.n_keys, table.arena_used
        if n1 <= n0:
            return
        dev = self.dev
        self._device_results(n1)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev.tdev))  # the piece's keys are in the table
        with torch.cuda.stream(self.ann):
            self.ann.wait_event(ev)
            # the table may re-allocate these while the side stream still reads them
            table.arena.record_stream(self.ann)
            table.key_ref.record_stream(self.ann)
            annot, hit = self.annot_d[n0:n1], self.hit_d[n0:n1]
            annot.fill_(0xFF)
            hit.fill_(-1)
            ks = KeySet(dev, table.arena, table.key_ref[n0:n1], n1 - n0)
            annotate_keys(dev, self.libs, ks, self.spike, out=(annot, hit))
            done = torch.cuda.Event()
            done.record(self.ann)
        if self.copy_out:
            with torch.cuda.stream(self.d2h):
                self.d2h.wait_event(done)
                self.to_host("arena", table.arena[w0:w1], w0, w0)
                self.to_host("key_ref", table.key_ref[n0:n1], n0, n0)
                self.to_host("annot", annot, n0, n0)
                self.to_host("hit", hit, n0, n0)
        self.n_done, self.w_done = n1, w1

    def results(self):
        """(annot uint8[n], hit int64[n]) on the device, valid on the current stream."""
        torch.cuda.current_stream(self.dev.tdev).wait_stream(self.ann)
        n = self.n_done
        if self.annot_d is None:
            e = torch.empty(0, dtype=torch.uint8, device=self.dev.tdev)
            return e, torch.empty(0, dtype=torch.int64, device=self.dev.tdev)
        return self.annot_d[:n], self.hit_d[:n]

    def finish(self, table: CollapseTable):
        """End of the sample: per-sample counts to the host; returns when every byte has arrived."""
        dev = self.dev
        ids, cnt = table.drain()
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev.tdev))
        with torch.cuda.stream(self.d2h):
            self.d2h.wait_event(ev)
            self.to_host("ids", ids, 0, 0)
            self.to_host("cnt", cnt, 0, 0)
        self.ann.synchronize()
        self.d2h.synchronize()
        return int(ids.numel())


def decode_hits(annot: np.ndarray, hit: np.ndarray):
    """(round, n_mismatch, ref_index, offset) numpy arrays from the packed hit words."""
    h = hit.view(np.uint64)
    return annot, (h >> np.uint64(56)).astype(np.int64), ((h >> np.uint64(28)) & np.uint64(0xFFFFFFF)).astype(np.int64), \
        (h & np.uint64(0xFFFFFFF)).astype(np.int64)


def load_libraries(args, ref_db: str, dev: Device) -> LibrarySet:
    key = (str(args.libraries_path), str(args.organism_name), str(ref_db), bool(args.spikeIn), dev.index)
    if key not in _LIB_CACHE:
        _LIB_CACHE[key] = LibrarySet.from_mirge_lib(dev, str(args.libraries_path), str(args.organism_name), str(ref_db),
                                                    bool(args.spikeIn))
    return _LIB_CACHE[key]


# per-round SAM files (alignPlusParse, manifoldAlign.py:20-45,57-62): -bam keeps rounds 0/8, 1, 4, 5, 6, 7; -trf rounds 2, 3
_SAM_BAM = {0: "miRge3_miRNA.sam", 8: "miRge3_miRNA.sam", 1: "miRge3_hairpin_miRNA.sam", 4: "miRge3_snorna.sam",
            5: "miRge3_rrna.sam", 6: "miRge3_ncrna_others.sam", 7: "miRge3_mrna.sam"}
_SAM_TRF = {2: "miRge3_tRNA.sam", 3: "miRge3_pre_tRNA.sam"}


def sam_rounds(args, spike: bool):
    """(round, SAM file name) of the rounds whose records the flags ask for, in the order they are appended."""
    want_bam, want_trf = bool(getattr(args, "bam_out", False)), bool(getattr(args, "tRNA_frag", False))
    out = []
    for rnd in range(10 if spike else 9):
        fname = (_SAM_BAM.get(rnd) if want_bam else None) or (_SAM_TRF.get(rnd) if want_trf else None)
        if fname is not None:
            out.append((rnd, fname))
    return out


def best_stratum_hits(dev: Device, lib, pol, keys: KeySet, ids: np.ndarray, hit_d: torch.Tensor):
    """All hits of the best stratum for the sequences ``ids`` of a -a --best --strata round: (row index into ids,
    hit word) pairs, unique, grouped by row, ascending hit word inside a row."""
    n = int(ids.size)
    if n == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.uint64)
    ids_d = torch.from_numpy(ids.astype(np.int32)).to(dev.tdev)
    counts = dev.zeros(n, torch.int32)
    call = lambda fill, offs, out: dev.check(dev.lib.mirge_annotate_allhits(
        dev.ctx, C.byref(lib.struct), C.byref(pol), C.byref(keys.struct), _ptr(ids_d), n, _ptr(hit_d), fill, _ptr(counts),
        _ptr(offs), _ptr(out), dev.stream()))
    call(0, None, None)
    offs = torch.cumsum(counts.to(torch.int64), 0) - counts.to(torch.int64)
    total = int((offs[-1] + counts[-1]).item())
    out = dev.empty(total, torch.int64)
    call(1, offs, out)
    dev.launches += 2
    rows = np.repeat(np.arange(n, dtype=np.int64), counts.cpu().numpy())
    words = out[:total].cpu().numpy().view(np.uint64)
    pairs = np.unique(np.stack([rows.astype(np.uint64), words], axis=1), axis=0)  # drops per-piece duplicates, sorts
    return pairs[:, 0].astype(np.int64), pairs[:, 1]


def _md_tag(query: str, ref_seg: str, seed: int):
    """(XA stratum, MD:Z string, NM) of an ungapped alignment, bowtie style."""
    q = np.frombuffer(query.upper().encode("latin-1"), dtype=np.uint8)
    r = np.frombuffer(ref_seg.upper().encode("latin-1"), dtype=np.uint8)
    acgt = (q == 65) | (q == 67) | (q == 71) | (q == 84)
    mis = np.nonzero(~((q == r) & acgt))[0]
    if mis.size == 0:
        return 0, str(len(query)), 0
    parts, prev = [], 0
    for p in mis.tolist():
        parts.append(str(p - prev))
        parts.append(ref_seg[p].upper())
        prev = p + 1
    parts.append(str(len(query) - prev))
    return int((mis < seed).sum()), "".join(parts), int(mis.size)


def round_query_text(seq: str, pol) -> str:
    """What bowtie aligns (and prints as SEQ) for ``seq`` in a round: round 3 strips the trailing T{3,} run
    (manifoldAlign.py:118-126), -5 / -3 trim the ends."""
    q = seq
    if pol.strip_polyT:
        e = len(q)
        while e > 0 and q[e - 1] == "T":
            e -= 1
        q = q[:e]
    return q[pol.trim5 : max(len(q) - pol.trim3, pol.trim5)]


SAM_SLICE_BYTES = 512 << 20  # device buffer of one fill launch of mirge_sam_format; a larger round is formatted in slices


def round_sam_pairs(dev: Device, lib, pol, keys: KeySet, ids: np.ndarray, hit_d: torch.Tensor):
    """(key id, hit word) of every SAM record of one round for the sequences ``ids`` (key ids of ``keys``, in the order
    the records are wanted), in the order bowtie prints them: the canonical hit of a -n / -v round; every hit of the best
    stratum of a -a round (2, 3), hit words descending inside a sequence so that the canonical pick comes last (the
    record the reference's parser keeps, manifoldAlign.py:50-56).  Returns (key ids int64 numpy, hit words int64 on the
    device)."""
    ids = np.asarray(ids, dtype=np.int64)
    if pol.round in _SAM_TRF:
        r_idx, words = best_stratum_hits(dev, lib, pol, keys, ids, hit_d)
        o = np.lexsort((np.iinfo(np.int64).max - words.astype(np.int64), r_idx))  # sequence ascending, hit descending
        return ids[r_idx[o]], torch.from_numpy(np.ascontiguousarray(words[o]).view(np.int64)).to(dev.tdev)
    return ids, hit_d[torch.from_numpy(ids).to(dev.tdev)]


def _sam_names(dev: Device, lib):
    """The library's reference names on the device (bytes back to back, int64 offsets), made once per library."""
    got = getattr(lib, "_sam_names", None)
    if got is None:
        enc = [nm.encode("utf-8") for nm in lib.names]
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        np.cumsum(np.fromiter((len(b) for b in enc), dtype=np.int64, count=len(enc)), out=off[1:])
        blob = torch.from_numpy(np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8).copy()).to(dev.tdev)
        got = lib._sam_names = (blob, torch.from_numpy(off).to(dev.tdev))
    return got


def sam_records(dev: Device, lib, pol, keys: KeySet, ids: np.ndarray, hits_d: torch.Tensor, slice_bytes: int = 0):
    """The bowtie SAM records of the (key id, hit word) pairs (ids[i], hits_d[i]), formatted on the device by
    mirge_sam_format (csrc/sam_format.cuh) in that order.  Yields (record bytes uint8, record lengths int64) on the
    host per slice of at most ``slice_bytes`` (SAM_SLICE_BYTES) bytes -- one record more when a single record is
    larger."""
    n = int(len(ids))
    if n == 0:
        return
    ids_d = torch.from_numpy(np.asarray(ids).astype(np.int32)).to(dev.tdev)
    hits_d = hits_d.to(torch.int64).contiguous()
    names, name_off = _sam_names(dev, lib)
    call = lambda fill, i0, i1, lens, offs, out: dev.check(dev.lib.mirge_sam_format(
        dev.ctx, C.byref(lib.struct), C.byref(pol), C.byref(keys.struct), _ptr(ids_d[i0:i1]), _ptr(hits_d[i0:i1]), i1 - i0,
        _ptr(names), _ptr(name_off), fill, _ptr(lens), _ptr(offs), _ptr(out), dev.stream()))
    lens = dev.empty(n, torch.int32)
    with dev.timed("sam_format"):
        call(0, 0, n, lens, None, None)
    dev.launches += 1
    lens64 = lens[:n].to(torch.int64)
    ends = torch.cumsum(lens64, 0)
    ends_h, lens_h = ends.cpu().numpy(), lens64.cpu().numpy()
    budget = int(slice_bytes or SAM_SLICE_BYTES)
    i0 = 0
    while i0 < n:
        base = int(ends_h[i0 - 1]) if i0 else 0
        i1 = max(i0 + 1, int(np.searchsorted(ends_h, base + budget, side="right")))
        out = dev.empty(int(ends_h[i1 - 1]) - base, torch.uint8)
        offs = ends[i0:i1] - lens64[i0:i1] - base
        with dev.timed("sam_format"):
            call(1, i0, i1, None, offs, out)
        dev.launches += 1
        yield out[: int(ends_h[i1 - 1]) - base].cpu().numpy(), lens_h[i0:i1]
        i0 = i1


def write_round_sam(path, dev: Device, lib, pol, keys: KeySet, ids: np.ndarray, hit_d: torch.Tensor, slice_bytes: int = 0):
    """Append the SAM records of one round (round_sam_pairs of the sequences ``ids``, in that order) to ``path``; the
    records are formatted on the device and copied to the host once per slice.  Returns (records, bytes) written."""
    rec_ids, rec_hits = round_sam_pairs(dev, lib, pol, keys, ids, hit_d)
    n_rec = n_bytes = 0
    with open(path, "ab") as fh:
        for chunk, lens in sam_records(dev, lib, pol, keys, rec_ids, rec_hits, slice_bytes):
            fh.write(memoryview(chunk))
            n_rec += int(lens.size)
            n_bytes += int(chunk.size)
    return n_rec, n_bytes


def write_sam_files(args, workDir, dev: Device, libs, keys: KeySet, annot: np.ndarray, key_of_row: Optional[np.ndarray],
                    hit_of_key: torch.Tensor, spike: bool):
    """The per-round SAM files for bamFmt.bow2bam (-bam) and the tRF block of summarize (-trf) that ``args`` asks for:
    records in the order bowtie prints them (input order = table order, round_sam_pairs inside a sequence), formatted
    on the device.  annot: annotation round of every table row; key_of_row: key id of every row (None: row = key id);
    hit_of_key: hit word of every key id, on the device."""
    pols = round_policies()
    for rnd, fname in sam_rounds(args, spike):
        rows = np.nonzero(annot == rnd)[0]
        if rows.size == 0:
            continue
        ids = rows if key_of_row is None else key_of_row[rows]
        write_round_sam(Path(workDir) / fname, dev, libs[ROUND_LIBS[rnd]], pols[rnd], keys, ids, hit_of_key)


def _filled_column(old: "pd.Series", rows: np.ndarray, names: np.ndarray, ref: np.ndarray):
    """The annotation column of a round: names[ref] at ``rows``, the old values elsewhere (manifoldAlign.py:17-18,55).
    A column that is still all '' -- what baking() hands over -- is built from codes + dictionary (Arrow dictionary
    decode for pandas' string dtype, one object take otherwise) instead of turning every cell into a Python object
    and back: the difference is seconds per round on tens of millions of rows."""
    n = len(old)
    fresh = n > 100_000 and not bool((old != "").any())
    if not fresh:
        col = old.to_numpy(dtype=object, copy=True)
        col[rows] = names[ref]
        return col
    codes = np.zeros(n, dtype=np.int32)
    codes[rows] = 1 + ref.astype(np.int32)
    ext = np.concatenate([np.array([""], dtype=object), names])
    if old.dtype == object:
        return ext[codes]
    import pandas as pd
    import pyarrow as pa

    arr = pa.DictionaryArray.from_arrays(pa.array(codes), pa.array(ext.tolist(), type=pa.large_string())).dictionary_decode()
    return pd.array(arr, dtype=old.dtype)


def _round_column_device(dev: Device, annot_d: torch.Tensor, ref_d: torch.Tensor, rnd: int, names, dtype):
    """The same column for pandas' Arrow-backed string dtype, assembled on the device: per-row name lengths -> running
    sum = the Arrow offsets buffer, name bytes gathered into the data buffer; two device-to-host copies and no pass over
    the rows on the host.  None when the round annotated nothing."""
    import pandas as pd
    import pyarrow as pa

    rows = torch.nonzero(annot_d == rnd).squeeze(1)
    if rows.numel() == 0:
        return None
    n = int(annot_d.numel())
    enc = [nm.encode("utf-8") for nm in names]
    name_len = torch.from_numpy(np.fromiter((len(b) for b in enc), dtype=np.int64, count=len(enc))).to(dev.tdev)
    name_off = torch.cumsum(name_len, 0) - name_len
    blob = torch.from_numpy(np.frombuffer(b"".join(enc) or b"\0", dtype=np.uint8).copy()).to(dev.tdev)
    ref_r = ref_d[rows].to(torch.int64)
    lens_r = name_len[ref_r]
    offsets = torch.zeros(n + 1, dtype=torch.int64, device=dev.tdev)
    offsets[rows + 1] = lens_r
    torch.cumsum(offsets, 0, out=offsets)
    total = int(offsets[-1].item())
    out_start = offsets[rows]
    src = torch.arange(total, device=dev.tdev, dtype=torch.int64) - torch.repeat_interleave(out_start - name_off[ref_r], lens_r)
    data = blob[src] if total else blob[:0]
    arr = pa.LargeStringArray.from_buffers(n, pa.py_buffer(offsets.cpu().numpy()), pa.py_buffer(data.cpu().numpy()))
    return pd.array(arr, dtype=dtype)


def _fill_rounds_device(pdDataFrame, dev: Device, annot_d: torch.Tensor, ref_d: torch.Tensor, libs, n_rounds: int) -> bool:
    """_fill_rounds with the columns built on the device; False (nothing done) unless the table is large and every
    annotation column is still the all-'' Arrow string column baking() hands over."""
    colnames = list(pdDataFrame.columns)
    n = len(pdDataFrame)
    if n < 1_000_000:
        return False
    for rnd in range(n_rounds):
        col = pdDataFrame[colnames[1 + rnd]]
        if col.dtype == object or not hasattr(col.array, "_pa_array") or bool((col != "").any()):
            return False
    for rnd in range(n_rounds):
        col = _round_column_device(dev, annot_d, ref_d, rnd, libs[ROUND_LIBS[rnd]].names, pdDataFrame[colnames[1 + rnd]].dtype)
        if col is not None:
            pdDataFrame[colnames[1 + rnd]] = col
    return True


def _fill_rounds(pdDataFrame, annot: np.ndarray, ref: np.ndarray, libs, n_rounds: int, threads: int = 0):
    """Columns 1 + round of every round that annotated something (manifoldAlign.py:17-18,55).  The rounds are independent
    (a sequence is annotated by one round), so large tables build their columns on a few threads: numpy and Arrow
    release the GIL for the passes over tens of millions of rows."""
    colnames = list(pdDataFrame.columns)

    def one(rnd):
        rows = np.nonzero(annot == rnd)[0]
        if rows.size == 0:
            return rnd, None
        names = np.asarray(libs[ROUND_LIBS[rnd]].names, dtype=object)
        return rnd, _filled_column(pdDataFrame[colnames[1 + rnd]], rows, names, ref[rows])

    rounds = list(range(n_rounds))
    if len(annot) > 1_000_000:
        from concurrent.futures import ThreadPoolExecutor

        with ThreadPoolExecutor(max_workers=max(1, min(len(rounds), threads or (os.cpu_count() or 4)))) as ex:
            built = list(ex.map(one, rounds))
    else:
        built = [one(r) for r in rounds]
    for rnd, col in built:
        if col is not None:
            pdDataFrame[colnames[1 + rnd]] = col


def _rows_match(cached, index, probes: int = 64) -> bool:
    """The key cache of a DataFrame is only used while its rows are still the ones baking() returned: first, last and a
    seeded sample of rows are decoded from the device table and compared with the index."""
    table, order = cached.table, cached.order
    n = len(index)
    if n == 0:
        return True
    rng = np.random.default_rng(12345)
    rows = np.unique(np.concatenate([[0, n - 1], rng.integers(0, n, size=min(probes, n))]))
    for i in rows.tolist():
        if table.export_keys(int(order[i]), 1)[0].decode("latin-1") != str(index[i]):
            return False
    return True


def bwtAlign(args, pdDataFrame, workDir, ref_db, libraries: Optional[LibrarySet] = None, device: Optional[Device] = None):
    """Same contract as the reference ``bwtAlign(args, pdDataFrame, workDir, ref_db)``
    (manifoldAlign.py:68-146): fills the annotation column of the first round that hits each
    sequence (column index 1 + round, manifoldAlign.py:17-18,55), sets annotFlag = 1 (:56), drops the
    'spike-in' column unless -spk (:137-138), fillna('') (:141) and logs to run.log (:83,144)."""
    begningTime = time.perf_counter()
    runlogFile = Path(workDir) / "run.log"
    outlog = open(str(runlogFile), "a+")
    if not getattr(args, "quiet", False):
        print("Alignment in progress ...")
    outlog.write("Alignment in progress ...\n")
    dev = device or get_device()
    libs = libraries or load_libraries(args, ref_db, dev)
    spike = bool(getattr(args, "spikeIn", False))
    annot_dv = hit_dv = None
    cached = pdDataFrame.attrs.get("_mirge_b200_keys")
    if cached is not None and getattr(cached.table, "dev", None) is dev and len(cached.order) == len(pdDataFrame) and \
            _rows_match(cached, pdDataFrame.index):
        # the DataFrame comes straight from baking(): its packed keys are still on the device (row i = key id order[i])
        table, order = cached.table, cached.order
        keys = KeySet.from_table(table)
        annot_all, hit_all = annotate_keys(dev, libs, keys, spike)
        sel = getattr(cached, "order_d", None)
        if sel is None:
            sel = torch.from_numpy(np.ascontiguousarray(order)).to(dev.tdev)
        annot_dv, hit_dv = annot_all[sel], hit_all[sel]
        annot = annot_dv.cpu().numpy()
        hit = None  # (copied only if the columns have to be built on the host)
        key_of_row, hit_of_key = order, hit_all
    else:
        seqs = pdDataFrame.index.to_numpy()
        keys = KeySet.from_strings(dev, list(seqs))
        annot_d, hit_d = annotate_keys(dev, libs, keys, spike)
        annot = annot_d.cpu().numpy()
        hit = hit_d.cpu().numpy()
        key_of_row, hit_of_key = None, hit_d  # key id = row
    colnames = list(pdDataFrame.columns)
    n_rounds = 10 if spike else 9
    on_device = False
    if annot_dv is not None:
        on_device = _fill_rounds_device(pdDataFrame, dev, annot_dv, (hit_dv >> 28) & 0xFFFFFFF, libs, n_rounds)
    if not on_device:
        if hit is None:
            hit = hit_dv.cpu().numpy()
        ref = ((hit.view(np.uint64) >> np.uint64(28)) & np.uint64(0xFFFFFFF)).astype(np.int64)  # decode_hits()[2]
        _fill_rounds(pdDataFrame, annot, ref, libs, n_rounds, int(getattr(args, "threads", 0) or 0))
    flag = pdDataFrame[colnames[0]].to_numpy(copy=True)
    flag[annot != 0xFF] = 1
    pdDataFrame[colnames[0]] = flag
    write_sam_files(args, workDir, dev, libs, keys, annot, key_of_row, hit_of_key, spike)
    finish = time.perf_counter()
    if not spike:
        pdDataFrame = pdDataFrame.drop(columns=["spike-in"])
    pdDataFrame = pdDataFrame.fillna("")
    if not getattr(args, "quiet", False):
        print(f"Alignment completed in {round(finish-begningTime, 4)} second(s)\n")
    outlog.write(f"Alignment completed in {round(finish-begningTime, 4)} second(s)\n")
    outlog.close()
    return pdDataFrame
