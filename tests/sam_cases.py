"""Inputs and oracle of the per-round SAM file tests (tests/test_gpu_sam.py, tests/multi_gpu_sam_check.py): libraries
whose tRNA sets hold exact and near duplicates (so the -a rounds 2 and 3 list several best-stratum hits per sequence)
and references with N; samples whose reads carry miRNA, isomiR, tRNA fragment, poly-T-tailed pre-tRNA and other
library inserts; and the SAM files the reference would write for a bwtAlign result, built with pyoracle.sam_line."""
import gzip
import os

import numpy as np

from oracle import pyoracle as po
from tests.test_gpu_annotate import make_libs
from tests.util import ILL

B = np.array(list("ACGT"))


def _sub(rng, s, k):
    s = list(s)
    for j in rng.choice(len(s), size=k, replace=False):
        s[j] = str(rng.choice([c for c in "ACGT" if c != s[j]]))
    return "".join(s)


def make_sam_libs(rng, scale=0.2):
    """make_libs plus, in both tRNA libraries, exact copies and one- and two-substitution variants of the first
    references (other names, so a best stratum spans several references) and an N in every fifth reference."""
    libs = make_libs(rng, scale)
    for k in ("mature_trna", "pre_trna"):
        names, seqs = libs[k]
        names, seqs = list(names), list(seqs)
        base = len(seqs)
        for i in range(min(6, base)):
            seqs.append(seqs[i])
            names.append("%s_dup%d" % (k, i))
            seqs.append(_sub(rng, seqs[i], 1 + i % 2))
            names.append("%s_var%d" % (k, i))
        for i in range(7, base, 5):
            p = int(rng.integers(len(seqs[i])))
            seqs[i] = seqs[i][:p] + "N" + seqs[i][p + 1:]
        libs[k] = (names, seqs)
    return libs


def insert(rng, libs):
    """One read insert: a library sequence or fragment of it, sometimes with a mismatch, isomiR ends or a T tail."""
    r = rng.random()
    if r < 0.35:
        m = libs["mirna"][1][int(rng.integers(min(12, len(libs["mirna"][1]))))]
        if rng.random() < 0.3:
            m = str(rng.choice(B)) + m + "".join(rng.choice(B, 2))
        return m
    key = "mature_trna" if r < 0.6 else "pre_trna" if r < 0.8 else str(rng.choice(["hairpin", "snorna", "rrna", "ncrna_others"]))
    seqs = libs[key][1]
    ref = seqs[int(rng.integers(min(8, len(seqs))))].replace("N", "A")
    L = int(rng.integers(18, 36))
    a = int(rng.integers(0, len(ref) - L + 1))
    s = ref[a : a + L]
    if rng.random() < 0.3:
        s = _sub(rng, s, 1)
    if key == "pre_trna" and rng.random() < 0.6:
        s = s + "T" * int(rng.integers(3, 7))
    return s


def write_samples(tmp, libs, n_samples=3, reads=1500, umi=False, seed=40):
    """FASTQ files (the second one gzipped) of reads insert + 3' adapter, 4-base UMI flanks with ``umi``; the last sample
    repeats a single read, so all its sequences have one owner.  Returns (paths, sample names)."""
    names = ["s%d" % i for i in range(n_samples)]
    files = []
    for i, n in enumerate(names):
        rng = np.random.default_rng(seed + i)
        one = insert(rng, libs) if i == n_samples - 1 else None
        recs = []
        for k in range(reads):
            ins = one or insert(rng, libs)
            pre = "".join(rng.choice(B, 4)) if umi else ""
            suf = "".join(rng.choice(B, 4)) if umi else ""
            s = (pre + ins + suf + ILL + "ACGTACGTACGTAC")[:70]
            recs.append("@r%d.%d\n%s\n+\n%s\n" % (i, k, s, "I" * len(s)))
        data = "".join(recs).encode()
        path = os.path.join(tmp, n + (".fastq.gz" if i == 1 else ".fastq"))
        if path.endswith(".gz"):
            with gzip.open(path, "wb") as fh:
                fh.write(data)
        else:
            with open(path, "wb") as fh:
                fh.write(data)
        files.append(path)
    return files, names


def round_hits(query, lib, rnd):
    """Hit words of the records bowtie prints for ``query`` in round ``rnd`` (exhaustive scan, pyoracle.hits): the
    canonical pick, or for the -a rounds 2 / 3 every hit of the best stratum, hit words descending."""
    hs = po.hits(query, lib, po.ROUND_POLICIES[rnd])
    if not hs:
        return []
    words = sorted(((h[0] << 56) | (h[1] << 28) | h[2]) for h in hs)
    if rnd in (2, 3):
        return sorted((w for w in words if (w >> 56) == (words[0] >> 56)), reverse=True)
    return words[:1]


def expected_sam_files(out, libs, bam: bool, trf: bool, spike: bool):
    """{file name: text} of the per-round SAM files for the bwtAlign result ``out`` (one round column filled per
    annotated row), from the exhaustive scan and pyoracle.sam_line, rows in table order."""
    from mirge_b200.manifoldAlign import round_query_text
    from mirge_b200.libraries import round_policies

    bam_files = {0: "miRge3_miRNA.sam", 8: "miRge3_miRNA.sam", 1: "miRge3_hairpin_miRNA.sam", 4: "miRge3_snorna.sam",
                 5: "miRge3_rrna.sam", 6: "miRge3_ncrna_others.sam", 7: "miRge3_mrna.sam"}
    trf_files = {2: "miRge3_tRNA.sam", 3: "miRge3_pre_tRNA.sam"}
    pols = round_policies()
    files = {}
    seqs = [str(s) for s in out.index]
    for rnd in range(10 if spike else 9):
        fname = (bam_files.get(rnd) if bam else None) or (trf_files.get(rnd) if trf else None)
        if fname is None:
            continue
        names, refs = libs[po.ROUND_LIBS[rnd]]
        lib = po.Library(list(names), [r.upper() for r in refs])
        col = out[po.ROUND_COLUMNS[rnd]].tolist()
        lines = []
        for s, c in zip(seqs, col):
            if c == "":
                continue
            q = round_query_text(s, pols[rnd])
            words = round_hits(q, lib, rnd)
            assert words and lib.names[(words[-1] >> 28) & 0xFFFFFFF] == c, (rnd, s, c)
            for w in words:
                r, off = (w >> 28) & 0xFFFFFFF, w & 0xFFFFFFF
                lines.append(po.sam_line(s, q, lib.names[r], lib.seqs[r], off, po.ROUND_POLICIES[rnd]) + "\n")
        if lines:
            files[fname] = files.get(fname, "") + "".join(lines)
    return files
