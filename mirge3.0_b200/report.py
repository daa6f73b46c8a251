"""Outputs that follow the annotation rounds: ``mapped.csv`` / ``unmapped.csv`` (mirge/__main__.py:164-173)
and the counters of ``annotation.report.csv`` / ``miR.Counts.csv`` that ``summarize`` derives from the mapped
table (mirge/libs/summary.py:677-770, 882-901, 1223-1224, 1275-1279).

The per-sample sums over the unique-sequence table (per-library read totals, exact-miRNA and isomiR reads per
miRNA) run on the device in one pass over the sample's (key id, count) pairs (csrc/report.cu); the
canonical-ratio filter and the name merging work on arrays of the size of the miRNA library and stay on the
host.  The reference's own ``summarize`` keeps working on the DataFrame ``bwtAlign`` returns; this module is
the same arithmetic without the pandas joins, for tables that do not fit a DataFrame comfortably."""
from __future__ import annotations

from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import pandas as pd
import torch

from .device import Device, MirgeError, _ptr
from .libraries import ROUND_COLUMNS, ROUND_LIBS, LibrarySet

REPORT_COLUMNS = ["Total Input Reads", "Trimmed Reads (all)", "Trimmed Reads (unique)", "All miRNA Reads", "Filtered miRNA Reads",
                  "Unique miRNAs", "Hairpin miRNAs", "mature tRNA Reads", "primary tRNA Reads", "snoRNA Reads", "rRNA Reads",
                  "ncRNA others", "mRNA Reads", "Spike-in", "Remaining Reads"]  # summary.py:897,901
_ROUND_OF = {"Hairpin miRNAs": 1, "mature tRNA Reads": 2, "primary tRNA Reads": 3, "snoRNA Reads": 4, "rRNA Reads": 5,
             "ncRNA others": 6, "mRNA Reads": 7, "Spike-in": 9}  # summary.py:686-691


def write_tables(pdDataFrame: pd.DataFrame, workDir) -> Tuple[pd.DataFrame, pd.DataFrame]:
    """__main__.py:164-165,170-173: split on annotFlag and write mapped.csv / unmapped.csv."""
    pdMapped = pdDataFrame[pdDataFrame.annotFlag.eq(1)]
    pdUnmapped = pdDataFrame[pdDataFrame.annotFlag.eq(0)]
    pdMapped.to_csv(Path(workDir) / "mapped.csv")
    pdUnmapped.to_csv(Path(workDir) / "unmapped.csv")
    return pdMapped, pdUnmapped


class SampleSums:
    """Device-side accumulators of one sample (summary.py:692-698,741-742)."""

    def __init__(self, dev: Device, n_mirna: int):
        self.dev, self.n_mirna = dev, int(n_mirna)
        self.round_sum = dev.zeros(10, torch.int64)
        self.can = dev.zeros(max(self.n_mirna, 1), torch.int64)
        self.iso = dev.zeros(max(self.n_mirna, 1), torch.int64)

    def add(self, annot: torch.Tensor, hit: torch.Tensor, ids: torch.Tensor, counts: torch.Tensor):
        """Accumulate the (key id, count) pairs of the sample; annot / hit are indexed by key id."""
        d = self.dev
        n = int(ids.numel())
        if n == 0:
            return
        if ids.dtype != torch.int32 or counts.dtype != torch.int32 or annot.dtype != torch.uint8 or hit.dtype != torch.int64:
            raise MirgeError("report: ids/counts must be int32, annot uint8, hit int64")
        d.check(d.lib.mirge_report_reduce(d.ctx, _ptr(annot), _ptr(hit), _ptr(ids), _ptr(counts), n, self.n_mirna,
                                          _ptr(self.round_sum), _ptr(self.can), _ptr(self.iso), d.stream()))
        d.launches += 1

    def host(self):
        return self.round_sum.cpu().numpy(), self.can[: self.n_mirna].cpu().numpy(), self.iso[: self.n_mirna].cpu().numpy()


def read_merges(path) -> Tuple[Dict[str, str], List[str]]:
    """<organism>_merges_<db>.csv (summary.py:705-714); a missing file means no merging (:715-716)."""
    member: Dict[str, str] = {}
    merged: List[str] = []
    try:
        with open(path, "r") as fh:
            for line in fh:
                c = line.strip().split(",")
                for item in c[1:]:
                    member[item] = c[0]
                merged.append(c[0])
    except FileNotFoundError:
        pass
    return member, merged


def canonical_filter(can: np.ndarray, iso: np.ndarray, ca_thr: float) -> np.ndarray:
    """mirge_can (summary.py:25-45), vectorised over the miRNAs of one sample."""
    x = can.astype(np.int64).copy()
    y = iso.astype(np.int64).copy()
    low = x < 2
    x[low] = 0
    y[low] = 0
    ratio = np.where(y > 0, x / np.maximum(y, 1), x.astype(np.float64))
    return np.where(ratio > ca_thr, x + y, 0)


def build_report(base_names: Sequence[str], sums: Sequence[Tuple[np.ndarray, np.ndarray, np.ndarray]], has_exact: np.ndarray,
                 mirna_names: Sequence[str], member: Dict[str, str], merged_names: Sequence[str], sampleReadCounts: Dict[str, int],
                 trimmedReadCounts: Dict[str, int], trimmedReadCountsUnique: Dict[str, int], ca_thr: float, spike_in: bool):
    """(annotation.report, miR.Counts, miR.RPM DataFrames) from the per-sample sums.  ``has_exact[ref]``: the miRNA
    has at least one exact-miRNA row in the mapped table (the rows of cann_collapse, summary.py:741)."""
    S = len(base_names)
    out_name = [member.get(n, n) for n in mirna_names]  # summary.py:750-752
    groups = sorted({out_name[r] for r in np.nonzero(has_exact)[0]})
    gidx = {n: i for i, n in enumerate(groups)}
    gof = np.array([gidx.get(out_name[r], -1) if has_exact[r] else -1 for r in range(len(mirna_names))], dtype=np.int64)
    grouped = np.zeros((len(groups), S), dtype=np.float64)
    rows = []
    for j, name in enumerate(base_names):
        round_sum, can, iso = sums[j]
        kept = canonical_filter(can, iso, ca_thr)
        sel = gof >= 0
        np.add.at(grouped[:, j], gof[sel], kept[sel].astype(np.float64))
        r = {"Total Input Reads": int(sampleReadCounts[name]), "Trimmed Reads (all)": int(trimmedReadCounts[name]),
             "Trimmed Reads (unique)": int(trimmedReadCountsUnique[name]),
             "All miRNA Reads": int(round_sum[0] + round_sum[8]),  # summary.py:764-766
             "Filtered miRNA Reads": int(grouped[:, j].sum()),  # :757-758
             "Unique miRNAs": int((grouped[:, j] > 0).sum())}  # :882-887
        for col, rnd in _ROUND_OF.items():
            if col == "Spike-in" and not spike_in:
                continue
            r[col] = int(round_sum[rnd])
        tosum = ["All miRNA Reads"] + [c for c in _ROUND_OF if c in r]
        r["Remaining Reads"] = r["Trimmed Reads (all)"] - sum(r[c] for c in tosum)  # :1224
        rows.append(r)
    cols = [c for c in REPORT_COLUMNS if spike_in or c != "Spike-in"]
    summary = pd.DataFrame(rows, index=pd.Index(list(base_names), name="Sample name(s)"), columns=cols).astype(int)
    # miR.Counts.csv (summary.py:774-797)
    names = list(merged_names)
    for srow in mirna_names:
        if "segs:" in srow:
            srow = srow.split(" ")[0]
        if srow not in member:
            names.append(srow)
    all_names = sorted(set(names) | set(groups))
    counts = np.zeros((len(all_names), S), dtype=np.float64)
    pos = {n: i for i, n in enumerate(all_names)}
    for n, i in gidx.items():
        counts[pos[n]] = grouped[i]
    mir_counts = pd.DataFrame(counts, index=pd.Index(all_names, name="miRNA"), columns=list(base_names))
    # miR.RPM.csv (summary.py:759,795,797): reads per million of the filtered miRNA reads, 4 decimals
    with np.errstate(divide="ignore", invalid="ignore"):
        rpm_g = np.round(grouped / grouped.sum(axis=0) * 1000000, 4)
    rpm = np.zeros((len(all_names), S), dtype=np.float64)
    for n, i in gidx.items():
        rpm[pos[n]] = rpm_g[i]
    mir_rpm = pd.DataFrame(np.nan_to_num(rpm, nan=0.0), index=pd.Index(all_names, name="miRNA"), columns=list(base_names))
    return summary, mir_counts, mir_rpm


def codes_from_dataframe(pdDataFrame: pd.DataFrame, libs: LibrarySet, spike_in: bool):
    """(annot uint8[n], hit int64[n]) of an annotated DataFrame: the round whose column is filled and the
    index of that name in the round's library -- the arrays annotate_keys leaves on the device."""
    n = len(pdDataFrame)
    annot = np.full(n, 0xFF, dtype=np.uint8)
    hit = np.full(n, -1, dtype=np.int64)
    for rnd in range(10 if spike_in else 9):
        col = pdDataFrame[ROUND_COLUMNS[rnd]].to_numpy(dtype=object)
        rows = np.nonzero(col != "")[0]
        if rows.size == 0:
            continue
        idx = {nm: i for i, nm in enumerate(libs[ROUND_LIBS[rnd]].names)}
        ref = np.fromiter((idx[v] for v in col[rows]), dtype=np.int64, count=rows.size)
        annot[rows] = rnd
        hit[rows] = ref << 28
    return annot, hit


def annotation_report(args, workDir, ref_db, base_names: Sequence[str], pdDataFrame: pd.DataFrame, sampleReadCounts, trimmedReadCounts,
                      trimmedReadCountsUnique, libraries: Optional[LibrarySet] = None, device: Optional[Device] = None,
                      write: bool = True):
    """annotation.report.csv, miR.Counts.csv and miR.RPM.csv from the DataFrame ``bwtAlign`` returned (same inputs
    as the reference's summarize(), summary.py:677).  Returns the three DataFrames."""
    from .manifoldAlign import get_device, load_libraries

    dev = device or get_device()
    libs = libraries or load_libraries(args, ref_db, dev)
    spike = bool(getattr(args, "spikeIn", False))
    annot, hit = codes_from_dataframe(pdDataFrame, libs, spike)
    n = len(pdDataFrame)
    annot_d = torch.from_numpy(annot).to(dev.tdev)
    hit_d = torch.from_numpy(hit).to(dev.tdev)
    ids_d = torch.arange(n, dtype=torch.int32, device=dev.tdev)
    samples = []
    for name in base_names:
        col = pdDataFrame[name].to_numpy()
        if n and int(col.max()) >= (1 << 31):
            raise MirgeError("report: a per-sequence count exceeds int32")
        samples.append((ids_d, torch.from_numpy(col.astype(np.int32)).to(dev.tdev)))
    return annotation_report_device(args, workDir, ref_db, base_names, annot_d, hit_d, samples, sampleReadCounts, trimmedReadCounts,
                                    trimmedReadCountsUnique, libraries=libs, device=dev, write=write)


def annotation_report_device(args, workDir, ref_db, base_names: Sequence[str], annot_d: torch.Tensor, hit_d: torch.Tensor, samples,
                             sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique, rows_d: Optional[torch.Tensor] = None,
                             libraries: Optional[LibrarySet] = None, device: Optional[Device] = None, write: bool = True):
    """annotation_report from device arrays instead of a DataFrame: annot_d (uint8) / hit_d (int64), the annotation
    round and hit word of every key id; ``samples``, each sample's (key ids int32, counts int32) on the device, taken
    as they are (annotation_report checks a DataFrame's counts against 2^31 before it calls this; a table's drained
    counts are int32 already); ``rows_d``, the key ids of the table's rows (None: every key id is a row).  Returns the
    three DataFrames."""
    from .manifoldAlign import get_device, load_libraries

    dev = device or get_device()
    libs = libraries or load_libraries(args, ref_db, dev)
    spike = bool(getattr(args, "spikeIn", False))
    mir = libs["mirna"]
    sums = []
    for ids_d, cnt_d in samples:
        ss = SampleSums(dev, mir.n_refs)
        ss.add(annot_d, hit_d, ids_d, cnt_d)
        sums.append(ss.host())
    a, h = (annot_d, hit_d) if rows_d is None else (annot_d[rows_d], hit_d[rows_d])
    has_exact = np.zeros(mir.n_refs, dtype=bool)
    has_exact[((h[a == 0] >> 28) & 0xFFFFFFF).cpu().numpy()] = True
    mfname = str(args.organism_name) + "_merges_" + str(ref_db) + ".csv"
    member, merged = read_merges(Path(args.libraries_path) / args.organism_name / "annotation.Libs" / mfname)
    summary, mir_counts, mir_rpm = build_report(base_names, sums, has_exact, mir.names, member, merged, sampleReadCounts,
                                                trimmedReadCounts, trimmedReadCountsUnique, float(getattr(args, "crThreshold", 0.1)), spike)
    if write:
        summary.to_csv(Path(workDir) / "annotation.report.csv")  # summary.py:1275-1279
        mir_counts.to_csv(Path(workDir) / "miR.Counts.csv")  # summary.py:796
        mir_rpm.to_csv(Path(workDir) / "miR.RPM.csv")  # summary.py:797
    return summary, mir_counts, mir_rpm
