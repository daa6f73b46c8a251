"""``baking`` -- drop-in for mirge/libs/digest.py:105 (same signature, same return tuple, same
run.log / _umiCounts.csv / .trim.collapse.fa side effects) that digests FASTQ on the GPU:
tokenise -> trim (cutadapt semantics) -> collapse -> optional UMI level -> sample x sequence matrix.

The reference fans 4 MB chunks out to a process pool running cutadapt modifiers per read
(digest.py:139-140,320-375) and merges Python dicts in the parent (digest.py:141-163); here each
batch of the stream goes through the kernels of csrc/ and never comes back to the host until the
final table is exported."""
from __future__ import annotations

import ctypes as C
import os
import time
from pathlib import Path
from typing import Dict, List, Optional, Tuple

import numpy as np
import pandas as pd
import torch

from . import ingest
from . import params as P
from .device import CollapseTable, Device, DigestEngine, FastqFormatError, MirgeError, _ptr
from .manifoldAlign import get_device

INITIAL_FLAGS = ["exact miRNA", "hairpin miRNA", "mature tRNA", "primary tRNA", "snoRNA", "rRNA", "ncrna others", "mRNA",
                 "isomiR miRNA", "spike-in"]  # digest.py:253

DEFAULT_BATCH_BYTES = 256 << 20


def default_count_mode() -> str:
    """HEAD counts after every modifier (digest.py:354-373); the released 0.1.x packages count once
    (SURVEY.md section 0 item 3).  HEAD is the default; MIRGE_B200_COUNT_MODE=release switches."""
    return os.environ.get("MIRGE_B200_COUNT_MODE", "head")


def _host_threads(args) -> Optional[int]:
    """Worker threads for reading / inflating input: the reference's ``-cpu`` / args.threads (digest.py:139)."""
    try:
        t = int(getattr(args, "threads", 0) or 0)
    except (TypeError, ValueError):
        t = 0
    return t if t > 0 else None


def _open_fastq(path: str, threads: Optional[int] = None):
    """One input file as a readinto() source: read / inflated on worker threads (ingest.py)."""
    return ingest.open_fastq(path, threads)


class HostStreamer:
    """Feeds a host byte stream (file object, bytes-like or pinned tensor) to the engine piece by piece.

    Pipeline: ``n_buf`` device buffers; the H2D copy of a piece goes to a fixed offset (``headroom``) of its
    buffer, so it does not depend on where the previous piece's last complete record ended and is enqueued
    ``n_buf - 1`` pieces ahead on its own stream -- the copy engine never waits for a kernel.  The tail of a
    piece that does not end on a record boundary is moved (device to device) in front of the next piece,
    into the headroom of that buffer.  ``on_piece(table)`` runs after every collapsed piece on the main
    stream (streamed annotation / D2H of the table's new keys)."""

    def __init__(self, eng: DigestEngine, batch_bytes: int = DEFAULT_BATCH_BYTES, max_record: int = 1 << 20, n_buf: int = 3):
        self.eng = eng
        self.dev = eng.dev
        self.batch = int(batch_bytes)
        self.n_buf = max(int(n_buf), 2)
        self.headroom = (int(max_record) + 64 + 255) & ~255
        self.d = [torch.empty(self.headroom + self.batch, dtype=torch.uint8, device=self.dev.tdev) for _ in range(self.n_buf)]
        self.h: List[Optional[torch.Tensor]] = [None] * self.n_buf  # pinned staging, only for readinto() sources
        self.h_busy: List[Optional[torch.cuda.Event]] = [None] * self.n_buf
        self.copy_stream = torch.cuda.Stream(device=self.dev.tdev)
        self.h2d_bytes = 0

    def _pieces(self, src):
        """Yield (pinned host tensor of <= batch bytes, staging index or -1) covering the stream, in order.
        A pinned torch tensor is sliced in place (no staging copy); anything with readinto() is staged
        through pinned buffers, each reused only after its previous H2D copy has completed."""
        if isinstance(src, torch.Tensor):
            if src.is_cuda or src.dtype != torch.uint8 or not src.is_pinned():
                raise MirgeError("host tensor source must be a pinned uint8 tensor")
            for pos in range(0, int(src.numel()), self.batch):
                yield src[pos : pos + self.batch], -1
            return
        cur = 0
        while True:
            if self.h[cur] is None:
                self.h[cur] = torch.empty(self.batch, dtype=torch.uint8).pin_memory()
            if self.h_busy[cur] is not None:
                self.h_busy[cur].synchronize()
            mv = memoryview(self.h[cur].numpy())
            got = 0
            while got < self.batch:
                k = src.readinto(mv[got:])
                if not k:
                    break
                got += k
            if got == 0:
                return
            yield self.h[cur][:got], cur
            if got < self.batch:
                return
            cur = (cur + 1) % self.n_buf

    def run(self, src, table: CollapseTable, on_piece=None, sharded=None) -> int:
        """Digest the whole stream into ``table``; returns the number of records parsed.  ``sharded``
        (distributed.ShardedCollapse, one process per GPU): the stream is this rank's share of the sample's reads; every
        piece's keys go to their owner ranks before the collapse, and ``table`` receives the keys this rank owns."""
        eng, dev, H = self.eng, self.dev, self.headroom
        main = torch.cuda.current_stream(dev.tdev)
        it = self._pieces(src)
        pending = []  # (buffer index, piece bytes, copy-done event)
        free_ev: List[Optional[torch.cuda.Event]] = [None] * self.n_buf
        state = {"k": 0, "done": False}

        def enqueue():
            if state["done"]:
                return
            nxt = next(it, None)
            if nxt is None:
                state["done"] = True
                return
            piece, hi = nxt
            b = state["k"] % self.n_buf
            n = int(piece.numel())
            with torch.cuda.stream(self.copy_stream):
                if free_ev[b] is not None:
                    self.copy_stream.wait_event(free_ev[b])  # kernels that read this buffer are done
                self.d[b][H : H + n].copy_(piece, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self.copy_stream)
            if hi >= 0:
                self.h_busy[hi] = ev
            pending.append((b, n, ev))
            self.h2d_bytes += n
            state["k"] += 1

        for _ in range(self.n_buf - 1):
            enqueue()
        n_records = 0
        more_any = True  # sharded: whether any rank has announced more input (unknown before this rank's first round)
        tail = 0  # bytes of the previous piece's incomplete last record, sitting just below the headroom mark
        while pending:
            b, n, ev = pending.pop(0)
            enqueue()
            final = not pending
            main.wait_event(ev)
            nbytes = tail + n
            view = self.d[b][H - tail : H + n]
            br = eng.trim_batch(view, nbytes, final, keep=False, table=None if sharded is not None else table)
            if not final:
                new_tail = nbytes - br.consumed
                if new_tail > H:
                    raise FastqFormatError("FASTQ record longer than %d bytes" % H)
                if br.n_records == 0 and new_tail == 0:
                    raise FastqFormatError("no complete FASTQ record in batch")
                if new_tail:
                    self.d[pending[0][0]][H - new_tail : H].copy_(view[br.consumed : nbytes])
                tail = new_tail
            if sharded is not None:
                more_any = sharded.round(table, br, not final, on_piece)
            else:
                eng.collapse_batch(table, br)
            fe = torch.cuda.Event()
            fe.record(main)
            free_ev[b] = fe
            n_records += br.n_records
            if sharded is None and on_piece is not None:
                on_piece(table)
        if sharded is not None:
            sharded.drain_rounds(table, more_any, on_piece)
        return n_records


class _BytesSource:
    def __init__(self, data):
        self.mv = memoryview(data).cast("B")
        self.pos = 0

    def readinto(self, out) -> int:
        k = min(len(out), len(self.mv) - self.pos)
        out[:k] = self.mv[self.pos : self.pos + k]
        self.pos += k
        return k


def umi_collapse(dev: Device, first: CollapseTable, ids: torch.Tensor, cnt: torch.Tensor, second: CollapseTable,
                 umi: Tuple[int, int], min_len: int, dedup: bool):
    """Second-level collapse (digest.py:164-205) of the drained first-level pairs into ``second``."""
    n = int(ids.numel())
    if n == 0:
        return
    second.check()
    second.reserve(n, int(first.arena_used))
    deferred = dev.empty(n, torch.int32)
    dev.check(dev.lib.mirge_umi_collapse(dev.ctx, C.byref(first.struct), _ptr(ids), _ptr(cnt), n, C.byref(second.struct),
                                         int(umi[0]), int(umi[1]), int(min_len), 1 if dedup else 0, _ptr(deferred), dev.stream()))
    dev.launches += 3
    second.check()


class SampleResult:
    """One sample's column of the matrix: (key id, count) pairs.  They stay on the device (``ids_d`` / ``counts_d``); the
    numpy views ``ids`` / ``counts`` are materialised on first use (the -tcf writer, the multi-GPU gather, tests)."""

    __slots__ = ("count", "trimmed", "unique", "_ids", "_counts", "ids_d", "counts_d", "rlen", "hist")

    def __init__(self):
        self._ids = self._counts = self.ids_d = self.counts_d = None

    @property
    def ids(self):
        if self._ids is None and self.ids_d is not None:
            self._ids = self.ids_d.cpu().numpy().astype(np.int64)
        return self._ids

    @ids.setter
    def ids(self, v):
        self._ids = v

    @property
    def counts(self):
        if self._counts is None and self.counts_d is not None:
            self._counts = self.counts_d.cpu().numpy().astype(np.int64)
        return self._counts

    @counts.setter
    def counts(self, v):
        self._counts = v


def digest_sample(eng: DigestEngine, source, table: CollapseTable, first_level: Optional[CollapseTable], umi_dedup: bool,
                  batch_bytes: int = DEFAULT_BATCH_BYTES, umi_csv: Optional[str] = None,
                  streamer: Optional[HostStreamer] = None) -> SampleResult:
    """One iteration of baking()'s per-sample loop (digest.py:133-217).  ``source`` is a device uint8
    tensor (already resident) or an object with readinto() / a bytes-like host buffer."""
    dev, cfg = eng.dev, eng.cfg
    umi = cfg.umi()
    target = first_level if umi is not None else table
    if isinstance(source, torch.Tensor) and source.is_cuda:
        count = eng.digest_device(source, target, batch_bytes)
    else:
        if not hasattr(source, "readinto") and not isinstance(source, torch.Tensor):
            source = _BytesSource(source)
        st = streamer or HostStreamer(eng, batch_bytes)
        count = st.run(source, target)
    res = SampleResult()
    res.count = count
    res.hist = np.zeros(0, dtype=np.int64)
    if umi is not None:
        ids1, cnt1 = first_level.drain()
        res.hist = cnt1.cpu().numpy().astype(np.int64)  # visual_treat['hist'] (digest.py:172,192)
        umi_collapse(dev, first_level, ids1, cnt1, table, umi, cfg.minimum_length, umi_dedup)
        if umi_dedup and umi_csv is not None:
            _write_umi_csv(umi_csv, first_level, ids1.cpu().numpy(), res.hist, umi, cfg.minimum_length)
        first_level.reset()
    ids, cnt = table.drain()
    res.ids_d, res.counts_d = ids, cnt
    res.trimmed = int(cnt.sum(dtype=torch.int64).item())  # digest.py:160-163 / 178-181 / 199-202
    res.unique = int(ids.numel())  # len(completeDict), digest.py:212
    return res


def _write_umi_csv(path: str, first: CollapseTable, ids: np.ndarray, counts: np.ndarray, umi: Tuple[int, int], min_len: int):
    """<sample>_umiCounts.csv (digest.py:185-205): header + one row per first-level key whose centre
    passes the length filter; opened in append mode like the reference (quirk 4)."""
    write_umi_csv_rows(path, umi_csv_rows(first.export_keys()[ids], counts, umi, min_len))


def umi_csv_rows(keys: np.ndarray, counts: np.ndarray, umi: Tuple[int, int], min_len: int) -> str:
    """The rows of <sample>_umiCounts.csv for first-level keys ``keys`` ('S' array) with their counts: centres shorter
    than ``min_len`` are left out."""
    f_, b_ = umi
    rows = []
    for k, c in zip(keys.tolist(), counts.tolist()):
        s = k.decode("latin-1")
        center = s[f_:-b_] if int(b_) != 0 else s[f_:]
        if len(center) >= int(min_len):
            rows.append(s[:f_] + s[-b_:] + "," + center + "," + str(c) + "\n")  # UMIParser incl. the b == 0 quirk
    return "".join(rows)


def write_umi_csv_rows(path: str, rows: str):
    """Header + ``rows`` appended to <sample>_umiCounts.csv (append mode like the reference, quirk 4)."""
    with open(path, "a+") as fh:
        fh.write("UMISeq" + "," + "transcriptSeq," + "UMICounts" + "\n")
        fh.write(rows)


def _no_keys():
    return None


class DeviceKeys:
    """What build_matrix leaves in DataFrame.attrs for bwtAlign: the table whose arena holds the packed keys and the
    key id of every row.  Not data: pickling the DataFrame (-spl / -rr, __main__.py:101,145) drops it."""

    def __init__(self, table, order, offsets=None, order_d=None):
        self.table, self.order, self.offsets, self.order_d = table, order, offsets, order_d

    @property
    def lens(self):
        """text length of every row (from the export's offsets; only the read-length histogram asks)"""
        return None if self.offsets is None else np.diff(self.offsets)

    def __reduce__(self):
        return (_no_keys, ())

    def __deepcopy__(self, memo):
        return self

    def __eq__(self, other):  # DataFrame.equals / comparisons of attrs never differ because of the cache
        return True

    def __hash__(self):
        return 0


ARROW_INDEX_MIN = int(os.environ.get("MIRGE_B200_ARROW_INDEX_MIN", str(2_000_000)))
MATRIX_DEVICE_BYTES = int(os.environ.get("MIRGE_B200_MATRIX_DEVICE_BYTES", str(16 << 30)))  # sample x sequence counts kept in HBM


def sequence_index(keys: np.ndarray) -> pd.Index:
    """The 'Sequence' index from an 'S' array of sequences (see sequence_index_packed)."""
    n = int(keys.shape[0])
    width = keys.dtype.itemsize
    mat = keys.view(np.uint8).reshape(n, width)
    lens = (mat != 0).sum(axis=1).astype(np.int64)  # sequences hold no NUL: the padding is the only zero
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    data = mat[np.arange(width, dtype=np.int64)[None, :] < lens[:, None]]
    return sequence_index_packed(offsets, data)


def sequence_index_packed(offsets: np.ndarray, data: np.ndarray) -> pd.Index:
    """The 'Sequence' index of the matrix from texts stored back to back.  Up to ARROW_INDEX_MIN rows: Python strings
    (object dtype, as the reference builds it).  Beyond: an Arrow-backed string index wrapped around the two buffers
    without creating a Python object per row -- tens of millions of str objects cost more than the whole device
    pipeline; element access, .str methods, to_csv and joins behave the same."""
    n = int(offsets.shape[0]) - 1
    if n < ARROW_INDEX_MIN or (data.size and int(data.max()) >= 128):
        blob = data.tobytes()
        off = offsets.tolist()
        return pd.Index([blob[off[i] : off[i + 1]].decode("latin-1") for i in range(n)], name="Sequence", dtype=object)
    import pyarrow as pa

    arr = pa.LargeStringArray.from_buffers(n, pa.py_buffer(np.ascontiguousarray(offsets, dtype=np.int64)),
                                           pa.py_buffer(np.ascontiguousarray(data)))
    return pd.Index(pd.arrays.ArrowStringArray(arr), name="Sequence")


def empty_flag_column(n: int):
    """A column of n empty strings with the dtype ``df.assign(col="")`` gives under the installed pandas (object before
    3.0, the Arrow-backed ``str`` dtype from 3.0 on) -- for the Arrow dtype one shared all-zero offsets buffer instead of
    n Python objects (``assign`` of ten such columns took 8 s for 39 M rows)."""
    dt = pd.DataFrame(index=[0]).assign(x="")["x"].dtype
    if dt == object:
        return np.full(n, "", dtype=object)
    import pyarrow as pa

    arr = pa.LargeStringArray.from_buffers(n, pa.py_buffer(np.zeros(n + 1, dtype=np.int64)), pa.py_buffer(b""))
    return pd.array(arr, dtype=dt)


def sample_columns(table: CollapseTable, samples: List[SampleResult], dtype):
    """(counts [samples, key ids] on the device, one contiguous row per sample; bool per key id, some sample counted
    it) from the samples' (key id, count) pairs."""
    cols_d = torch.zeros((len(samples), int(table.n_keys)), dtype=dtype, device=table.dev.tdev)
    for j, s in enumerate(samples):
        cols_d[j, s.ids_d.long()] = s.counts_d.to(dtype)
    return cols_d, (cols_d != 0).any(dim=0)


def build_matrix(table: CollapseTable, samples: List[SampleResult], names: List[str]) -> pd.DataFrame:
    """digest.py:237-261: unique sequences x samples, rows in lexicographic order (what pandas' outer
    join produces for > 1 sample; the single-sample order of the reference is not deterministic).  Columns as the
    reference leaves them (digest.py:253-256): annotFlag (int), the ten annotation columns (''), the samples."""
    n = int(table.n_keys)
    on_device = n > 0 and all(s.ids_d is not None for s in samples) and hasattr(table, "export_sorted_device") and \
        8 * n * max(len(samples), 1) <= MATRIX_DEVICE_BYTES
    if on_device:
        # the columns are scattered, selected and ordered on the device; the host sees each of them once, finished
        cols_d, seen_d = sample_columns(table, samples, torch.int64)
        perm_d, offsets_d, data_d = table.export_sorted_device(seen_d)
        order, offsets, data = perm_d.cpu().numpy(), offsets_d.cpu().numpy(), data_d.cpu().numpy()
        del offsets_d, data_d
        column = lambda j: cols_d[j][perm_d].cpu().numpy()
    else:
        perm_d = None
        cols = np.zeros((len(samples), n), dtype=np.int64)
        for j, s in enumerate(samples):
            cols[j, s.ids] = s.counts
        seen = cols.any(axis=0) if n else np.zeros(0, dtype=bool)
        # order, selection and the packed texts come from the device (CollapseTable.export_sorted)
        order, offsets, data = table.export_sorted(seen)
        column = lambda j: cols[j][order]
    index = sequence_index_packed(offsets, data)
    m = int(order.shape[0])
    empty = empty_flag_column(m)
    frame = {"annotFlag": np.zeros(m, dtype=np.dtype(int))}
    frame.update((f, empty) for f in INITIAL_FLAGS)
    df = pd.DataFrame(frame, index=index, copy=False)
    for j, name in enumerate(names):
        df[name] = column(j)
    if not len(names):
        df = df.reindex(columns=["annotFlag"] + INITIAL_FLAGS)
    # the packed keys stay on the device: bwtAlign finds them here instead of re-encoding every index string
    # (row i of the DataFrame = key id order[i] of the table); the text lengths serve the read-length histogram
    df.attrs["_mirge_b200_keys"] = DeviceKeys(table, order, offsets, perm_d)
    return df


def baking(args, inFileArray, inFileBaseArray, workDir, device: Optional[Device] = None, count_mode: Optional[str] = None,
           batch_bytes: int = DEFAULT_BATCH_BYTES, keep_table: bool = False):
    """Same contract as the reference ``baking(args, inFileArray, inFileBaseArray, workDir)``:
    returns (complete_set DataFrame, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique)."""
    begningTime = time.perf_counter()
    dev = device or get_device()
    runlogFile = Path(workDir) / "run.log"
    outlog = open(str(runlogFile), "a+")
    quiet = bool(getattr(args, "quiet", False))
    table, results, umi, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique = digest_samples(
        args, inFileArray, inFileBaseArray, workDir, dev, outlog, quiet, count_mode, batch_bytes)
    finish3 = time.perf_counter()
    complete_set = build_matrix(table, results, list(inFileBaseArray))
    finish4 = time.perf_counter()
    log_line(outlog, quiet, f"Matrix creation finished in {round(finish4-finish3, 4)} second(s)\n")
    names = list(inFileBaseArray)
    _write_histograms(workDir, lambda: _frame_lens(complete_set), lambda j: complete_set[names[j]].to_numpy() > 0, results, names,
                      umi)
    EndTime = time.perf_counter()
    log_line(outlog, quiet, f"Data pre-processing completed in {round(EndTime-begningTime, 4)} second(s)\n",
             f"\nData pre-processing completed in {round(EndTime-begningTime, 4)} second(s)\n\n")
    outlog.close()
    if keep_table:
        return complete_set, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique, table
    return (complete_set, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique)


def log_line(outlog, quiet: bool, screen: str, file: Optional[str] = None):
    """One progress line: print(screen) unless -quiet; ``file`` to run.log as it is (default: ``screen`` ending in one
    newline)."""
    if not quiet:
        print(screen)
    outlog.write(screen.rstrip("\n") + "\n" if file is None else file)


def digest_samples(args, inFileArray, inFileBaseArray, workDir, dev: Device, outlog, quiet: bool, count_mode: Optional[str] = None,
                   batch_bytes: int = DEFAULT_BATCH_BYTES):
    """baking()'s per-sample loop (digest.py:133-235): every file digested into one table, the counters, the -tcf /
    -umi -udd side files and the per-sample log lines.  Returns (table, [SampleResult], umi, sampleReadCounts,
    trimmedReadCounts, trimmedReadCountsUnique)."""
    cfg = P.TrimConfig.from_args(args, count_mode or default_count_mode())
    eng = DigestEngine(dev, cfg)
    umi = cfg.umi()
    table = CollapseTable(dev, min_keys=1 << 20)
    first_level = CollapseTable(dev, min_keys=1 << 20) if umi is not None else None
    streamer = HostStreamer(eng, batch_bytes)
    sampleReadCounts: Dict[str, int] = {}
    trimmedReadCounts: Dict[str, int] = {}
    trimmedReadCountsUnique: Dict[str, int] = {}
    results: List[SampleResult] = []
    # the files of the run are read (and inflated) ahead of the sample being digested, on args.threads workers
    readahead = ingest.SampleReadahead([str(p) for p in inFileArray], threads=_host_threads(args))
    for index, FQfile in enumerate(inFileArray):
        start = time.perf_counter()
        base = inFileBaseArray[index]
        umi_csv = str(Path(workDir) / (base + "_umiCounts.csv")) if (umi is not None and getattr(args, "umiDedup", False)) else None
        try:
            with readahead.open(index) as f:
                res = digest_sample(eng, f, table, first_level, bool(getattr(args, "umiDedup", False)), batch_bytes, umi_csv, streamer)
        except BaseException:
            readahead.close()
            raise
        results.append(res)
        sampleReadCounts[base] = res.count
        trimmedReadCounts[base] = res.trimmed
        trimmedReadCountsUnique[base] = res.unique
        finish2 = time.perf_counter()
        log_line(outlog, quiet, f"Cutadapt finished for file {base} in {round(finish2-start, 4)} second(s)")
        if getattr(args, "tcf_out", False):
            write_tcf(workDir, base, table, res)
        finish3 = time.perf_counter()
        log_line(outlog, quiet, f"Collapsing finished for file {base} in {round(finish3-finish2, 4)} second(s)\n")
    readahead.close()
    return table, results, umi, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique


def write_tcf(workDir, base, table: CollapseTable, res: SampleResult):
    """``<sample>.trim.collapse.fa`` (digest.py:226-235): the sample's sequences by descending count (stable)."""
    write_tcf_rows(workDir, base, table.export_keys()[res.ids], res.counts)


def write_tcf_rows(workDir, base, keys: np.ndarray, counts: np.ndarray):
    """``<sample>.trim.collapse.fa`` from the sample's sequences ``keys`` ('S' array) and their counts: by descending
    count (stable)."""
    order = np.argsort(-counts, kind="stable")
    with open(Path(workDir) / (str(base) + ".trim.collapse.fa"), "w") as fo:
        for hc, j in enumerate(order.tolist(), 1):
            fo.write(">seq" + str(hc) + "_" + str(int(counts[j])) + "\n")
            fo.write(keys[j].decode("latin-1") + "\n")


def _frame_lens(df: pd.DataFrame) -> np.ndarray:
    """Text length of every row of a frame from build_matrix (the export's offsets), else of its index."""
    cached = df.attrs.get("_mirge_b200_keys")
    if cached is not None and cached.offsets is not None and len(cached.offsets) == len(df) + 1:
        return cached.lens
    return df.index.str.len().to_numpy()


def _write_histograms(workDir, lens, present, results: List[SampleResult], names: List[str], umi):
    """index_data.js read-length / UMI histograms (digest.py:270-295) through the reference's own
    FormatJS when miRge is importable.  ``lens()``: the text length of every row of the table; ``present(j)``: bool
    per row, sample j counted it (both called only when the histograms are written).  Deviation (DESIGN.md): the
    reference appends one length per *chunk-unique* key (digest.py:146-157), which depends on its 4 MB chunk boundaries;
    here every sample-unique key contributes once."""
    try:
        from mirge.classes.exportHTML import FormatJS  # the reference's visualisation writer
    except Exception:
        return
    histData = FormatJS(workDir)
    lens = lens()
    for div_idnum, (name, res) in enumerate(zip(names, results), 1):
        val = lens[present(div_idnum - 1)]
        if val.size == 0:
            continue
        maxVal, minVal = int(val.max()), int(val.min())
        if maxVal > minVal:
            hist, bins = np.histogram(val, bins=(maxVal - minVal))
            histData.readLenDist("readLengthID_" + str(div_idnum), name, str(hist.tolist()), str(list(bins)))
        if umi is not None and res.hist.size:
            maxVal, minVal = int(res.hist.max()), int(res.hist.min())
            if maxVal > minVal:
                hist, bins = np.histogram(res.hist, bins=(maxVal - minVal))
                histData.sampleUMIDist("umiDivID_" + str(div_idnum), name, str(hist.tolist()), str(bins.tolist()))
