"""A miRge run's files written straight from the device table, without a DataFrame of it.

``baking`` + ``bwtAlign`` hand the sequence table over as a pandas DataFrame, and ``report.write_tables`` then writes
``mapped.csv`` / ``unmapped.csv`` with ``DataFrame.to_csv``: on tens of millions of rows both cost far more than the
device pipeline.  ``run_to_files`` goes from the FASTQ files to the same files, byte for byte: the table rows are
formatted on the device (``mirge_table_csv_format``, csrc/csv_format.cuh) from the packed keys, the annotation and
the sample x key count matrix, and copied to the host a slice at a time while a host thread writes the previous slice.
``write_table_csv`` is that writer on its own, for any selection of a table's rows."""
from __future__ import annotations

import ctypes as C
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path
from typing import Optional, Sequence

import torch

from . import digest as DG
from . import report as RP
from .device import Device, MirgeError, _ptr
from .libraries import ROUND_COLUMNS, ROUND_LIBS, LibrarySet
from .manifoldAlign import KeySet, annotate_keys, get_device, load_libraries, sam_rounds, write_sam_files

CSV_SLICE_BYTES = 64 << 20  # text of one fill launch: the device buffer and each of the two pinned host buffers


def csv_field(s: str) -> str:
    """``s`` as csv.QUOTE_MINIMAL (DataFrame.to_csv) writes it: in double quotes when it holds ',', '"', CR or LF,
    inner '"' doubled."""
    if any(c in s for c in ',"\r\n'):
        return '"' + s.replace('"', '""') + '"'
    return s


def table_csv_header(sample_names: Sequence[str], n_cols: int) -> bytes:
    """The header line to_csv writes for the table: index label, annotFlag, the first ``n_cols`` annotation columns,
    the samples."""
    cols = ["Sequence", "annotFlag"] + ROUND_COLUMNS[:n_cols] + [str(s) for s in sample_names]
    return (",".join(csv_field(c) for c in cols) + "\n").encode("utf-8")


def _column_names(dev: Device, libs: LibrarySet, n_cols: int):
    """(names uint8, offsets int64, round base int32) on the device: every round's reference names as finished CSV
    fields (UTF-8, quoted as to_csv quotes them), each library once; reference r of round c is field
    round_base[c] + r.  Made once per library set and column count."""
    cache = getattr(libs, "_csv_names", None)
    if cache is None:
        cache = libs._csv_names = {}
    got = cache.get(n_cols)
    if got is None:
        fields, base, placed = [], [], {}
        for c in range(n_cols):
            key = ROUND_LIBS[c]
            if key not in placed:
                placed[key] = len(fields)
                fields += [csv_field(nm).encode("utf-8") for nm in libs[key].names]
            base.append(placed[key])
        lens = torch.tensor([len(f) for f in fields], dtype=torch.int64)
        off = torch.zeros(len(fields) + 1, dtype=torch.int64)
        torch.cumsum(lens, 0, out=off[1:])
        blob = torch.frombuffer(bytearray(b"".join(fields) or b"\0"), dtype=torch.uint8)
        got = cache[n_cols] = (blob.to(dev.tdev), off.to(dev.tdev), torch.tensor(base, dtype=torch.int32).to(dev.tdev))
    return got


def _slices(ends: torch.Tensor, budget: int):
    """(first row, end row, first byte, end byte) of consecutive slices whose text fits ``budget`` bytes, cut from the
    rows' end offsets on the device (two scalar reads per slice; copying the offsets to the host instead cost more than
    all of them at the default slice size); a slice holds at least one row."""
    n, i0, base, out = int(ends.numel()), 0, 0, []
    while i0 < n:
        i1 = max(i0 + 1, int(torch.searchsorted(ends, base + budget, right=True).item()))
        end = int(ends[i1 - 1].item())
        out.append((i0, i1, base, end))
        i0, base = i1, end
    return out


def _write_when_copied(fh, done: torch.cuda.Event, buf: torch.Tensor, nbytes: int):
    done.synchronize()
    fh.write(memoryview(buf.numpy())[:nbytes])


def write_table_csv(path, dev: Device, table, rows_d: torch.Tensor, counts_d: Optional[torch.Tensor], sample_names: Sequence[str],
                    annot_d: Optional[torch.Tensor] = None, hit_d: Optional[torch.Tensor] = None, libs: Optional[LibrarySet] = None,
                    spike_in: bool = False, slice_bytes: int = CSV_SLICE_BYTES):
    """Write the rows ``rows_d`` (key ids of ``table``, a CollapseTable or KeySet, in output order) to ``path`` as
    DataFrame.to_csv writes them: the frame bwtAlign returns when annot_d / hit_d (annotation round / hit word by key id)
    and libs are given -- 9 annotation columns, 10 with ``spike_in`` --, else the unannotated frame baking returns (10
    empty columns).  counts_d: the [samples, key ids] count matrix (int32, read as uint32).  The text is formatted on
    the device in slices of about ``slice_bytes`` and written from a host thread while the next slice is formatted, so
    the text never needs more than two slices of device and pinned host memory; besides that, each row costs 16 bytes
    on the device (its key id as int32, its length, its end offset) and nothing on the host.  Returns (rows, bytes)
    written."""
    annotated = annot_d is not None
    if annotated and (hit_d is None or libs is None):
        raise MirgeError("table_csv: an annotated table needs hit words and libraries")
    n_cols = 10 if spike_in or not annotated else 9
    S = len(sample_names)
    header = table_csv_header(sample_names, n_cols)
    rows_d = rows_d.to(torch.int32).contiguous()
    n = int(rows_d.numel())
    counts = stride = None
    if S:
        counts = counts_d.to(torch.int32).contiguous()
        if counts.dim() != 2 or counts.shape[0] != S:
            raise MirgeError("table_csv: counts must be [samples, key ids]")
        stride = int(counts.shape[1])
    names = name_off = round_base = None
    if annotated:
        annot_d, hit_d = annot_d.to(torch.uint8).contiguous(), hit_d.to(torch.int64).contiguous()
        names, name_off, round_base = _column_names(dev, libs, n_cols)
    call = lambda fill, i0, i1, lens, offs, out: dev.check(dev.lib.mirge_table_csv_format(
        dev.ctx, C.byref(table.struct), _ptr(rows_d[i0:i1]), i1 - i0, _ptr(annot_d), _ptr(hit_d), _ptr(names), _ptr(name_off),
        _ptr(round_base), n_cols, _ptr(counts), S, stride or 0, fill, _ptr(lens), _ptr(offs), _ptr(out), dev.stream()))
    with open(path, "wb") as fh:
        fh.write(header)
        if n == 0:
            return 0, len(header)
        lens = dev.empty(n, torch.int32)
        with dev.timed("csv_format"):
            call(0, 0, n, lens, None, None)
        dev.launches += 1
        ends_d = torch.cumsum(lens[:n], 0, dtype=torch.int64)
        slices = _slices(ends_d, max(int(slice_bytes), 1))
        cap = max(e - b for _, _, b, e in slices)
        d_buf = [dev.empty(cap, torch.uint8) for _ in range(min(2, len(slices)))]
        h_buf = [torch.empty(cap, dtype=torch.uint8).pin_memory() for _ in d_buf]
        pending = [None] * len(d_buf)
        stream = torch.cuda.current_stream(dev.tdev)
        with ThreadPoolExecutor(max_workers=1) as writer:
            for k, (i0, i1, base, end) in enumerate(slices):
                b = k % len(d_buf)
                if pending[b] is not None:
                    pending[b].result()  # the host buffer's previous slice is in the file
                offs = ends_d[i0:i1] - lens[i0:i1] - base  # the slice's row offsets, relative to its first byte
                with dev.timed("csv_format"):
                    call(1, i0, i1, None, offs, d_buf[b])
                dev.launches += 1
                h_buf[b][: end - base].copy_(d_buf[b][: end - base], non_blocking=True)
                done = torch.cuda.Event()
                done.record(stream)
                pending[b] = writer.submit(_write_when_copied, fh, done, h_buf[b], end - base)
            for p in pending:
                p.result()
        return n, len(header) + slices[-1][3]


def run_to_files(args, inFileArray, inFileBaseArray, workDir, ref_db, device: Optional[Device] = None,
                 libraries: Optional[LibrarySet] = None, batch_bytes: int = DG.DEFAULT_BATCH_BYTES, count_mode: Optional[str] = None,
                 slice_bytes: int = CSV_SLICE_BYTES):
    """FASTQ files to miRge's output files with no DataFrame of the sequence table: writes what
    ``baking`` -> ``bwtAlign`` -> ``report.write_tables`` -> ``report.annotation_report`` write, with the same bytes --
    mapped.csv, unmapped.csv, annotation.report.csv, miR.Counts.csv, miR.RPM.csv, the per-round SAM files of -bam /
    -trf, <sample>.trim.collapse.fa of -tcf, <sample>_umiCounts.csv of -umi -udd, the index_data.js histograms when the
    reference's FormatJS is importable, and the run.log / stdout lines of baking and bwtAlign.  Rows are build_matrix's
    (keys some sample counted, in bytewise order of their text), split on the annotation on the device.  Returns
    (sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique)."""
    begningTime = time.perf_counter()
    dev = device or get_device()
    names = list(inFileBaseArray)
    quiet = bool(getattr(args, "quiet", False))
    runlog = str(Path(workDir) / "run.log")
    # baking: digest, matrix, histograms
    with open(runlog, "a+") as outlog:
        table, results, umi, src, trc, tru = DG.digest_samples(args, inFileArray, inFileBaseArray, workDir, dev, outlog, quiet,
                                                               count_mode, batch_bytes)
        finish3 = time.perf_counter()
        if 4 * int(table.n_keys) * max(len(results), 1) > DG.MATRIX_DEVICE_BYTES:
            raise MirgeError("run_to_files: the %d x %d sample x sequence count matrix (4 bytes a cell) exceeds "
                             "MIRGE_B200_MATRIX_DEVICE_BYTES (%d); baking + bwtAlign build it on the host"
                             % (len(results), int(table.n_keys), DG.MATRIX_DEVICE_BYTES))
        cols_d, seen_d = DG.sample_columns(table, results, torch.int32)
        perm_d, offsets_d, _ = table.export_sorted_device(seen_d)
        finish4 = time.perf_counter()
        DG.log_line(outlog, quiet, f"Matrix creation finished in {round(finish4-finish3, 4)} second(s)\n")
        DG._write_histograms(workDir, lambda: torch.diff(offsets_d).cpu().numpy(), lambda j: (cols_d[j][perm_d] != 0).cpu().numpy(),
                             results, names, umi)
        EndTime = time.perf_counter()
        DG.log_line(outlog, quiet, f"Data pre-processing completed in {round(EndTime-begningTime, 4)} second(s)\n",
                    f"\nData pre-processing completed in {round(EndTime-begningTime, 4)} second(s)\n\n")
    # bwtAlign: annotation rounds and SAM files
    begningTime = time.perf_counter()
    with open(runlog, "a+") as outlog:
        DG.log_line(outlog, quiet, "Alignment in progress ...")
        libs = libraries or load_libraries(args, ref_db, dev)
        spike = bool(getattr(args, "spikeIn", False))
        keys = KeySet.from_table(table)
        annot_d, hit_d = annotate_keys(dev, libs, keys, spike)
        annot_rows_d = annot_d[perm_d]
        if sam_rounds(args, spike):
            write_sam_files(args, workDir, dev, libs, keys, annot_rows_d.cpu().numpy(), perm_d.cpu().numpy(), hit_d, spike)
        finish = time.perf_counter()
        DG.log_line(outlog, quiet, f"Alignment completed in {round(finish-begningTime, 4)} second(s)\n")
    # write_tables + annotation_report
    mapped = annot_rows_d != 0xFF
    for fname, rows_d in (("mapped.csv", perm_d[mapped]), ("unmapped.csv", perm_d[~mapped])):
        write_table_csv(Path(workDir) / fname, dev, table, rows_d, cols_d, names, annot_d, hit_d, libs, spike, slice_bytes)
    RP.annotation_report_device(args, workDir, ref_db, names, annot_d, hit_d, [(r.ids_d, r.counts_d) for r in results], src, trc, tru,
                                rows_d=perm_d, libraries=libs, device=dev)
    return src, trc, tru
