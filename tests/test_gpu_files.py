"""outputs.run_to_files / write_table_csv (csrc/csv_format.cuh formatted on the device) against the files the reference
wrote (tests/golden/ref_case1..6) and, file for file and byte for byte, against the DataFrame path in the same process:
baking -> bwtAlign -> report.write_tables -> report.annotation_report.  Synthetic runs: several samples, library names
that need quoting, reads carrying ',', '"' and bytes >= 0x80, slices small enough that most rows are longer than a
slice, a table above 1 M rows (bwtAlign's device-built columns), and an empty table."""
import gzip
import os
import re

import numpy as np
import pytest

from tests.sam_cases import make_sam_libs, write_samples
from tests.test_gpu_annotate import write_lib_dir
from tests.test_reference_golden import CASE, DB, DIGEST_CASES, ORG, SAMPLES, golden, load_digest_case, sorted_lines, tcf_pairs
from tests.util import ILL, make_args

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

TABLES = ("mapped.csv", "unmapped.csv", "annotation.report.csv", "miR.Counts.csv", "miR.RPM.csv")


@pytest.fixture(scope="module")
def dev():
    from mirge_b200 import device as D

    return D.Device(0)


def dataframe_path(args, files, names, work, dev, ref_db=DB, batch_bytes=150_000):
    from mirge_b200 import digest as DG
    from mirge_b200 import manifoldAlign as MA
    from mirge_b200 import report as RP

    os.makedirs(work, exist_ok=True)
    df, src, trc, tru = DG.baking(args, files, names, work, device=dev, batch_bytes=batch_bytes)
    out = MA.bwtAlign(args, df, work, ref_db, device=dev)
    RP.write_tables(out, work)
    RP.annotation_report(args, work, ref_db, names, out, src, trc, tru, device=dev)
    return src, trc, tru


def files_path(args, files, names, work, dev, ref_db=DB, batch_bytes=150_000, **kw):
    from mirge_b200 import outputs as O

    os.makedirs(work, exist_ok=True)
    return O.run_to_files(args, files, names, work, ref_db, device=dev, batch_bytes=batch_bytes, **kw)


def timeless(text: str) -> str:
    return re.sub(r"in [0-9.e+-]+ second", "in T second", text)


def same_side_file(a, b, f):
    """The order of equal counts in .trim.collapse.fa, and of the rows of _umiCounts.csv, follows the order keys left
    the hash table, which two runs need not share (as two runs of the reference need not)."""
    pa, pb = os.path.join(a, f), os.path.join(b, f)
    if f.endswith(".trim.collapse.fa"):
        return tcf_pairs(pa) == tcf_pairs(pb)
    return open(pa).readline() == open(pb).readline() and sorted_lines(pa) == sorted_lines(pb)


def same_outputs(a, b):
    """Every file of work directory a equals the one of b (run.log up to its timings, side files up to the order of
    ties); returns the file names."""
    fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
    assert fa == fb
    for f in fa:
        if f.endswith((".trim.collapse.fa", "_umiCounts.csv")):
            assert same_side_file(a, b, f), f
            continue
        x, y = open(os.path.join(a, f), "rb").read(), open(os.path.join(b, f), "rb").read()
        if f == "run.log":
            x, y = timeless(x.decode()), timeless(y.decode())
        assert x == y, f
    return fa


def case1_args(**kw):
    return make_args(libraries_path=os.path.join(CASE, "lib"), organism_name=ORG, quality_cutoff="20", crThreshold="0.1", **kw)


def test_case1_files_equal_the_reference(dev, tmp_path):
    files = [os.path.join(CASE, s + ".fastq.gz") for s in SAMPLES]
    args = case1_args(spikeIn=True, bam_out=True, tRNA_frag=True)
    src, trc, tru = files_path(args, files, SAMPLES, str(tmp_path / "f"), dev, slice_bytes=8192)
    assert src["sampleA"] == 2500
    for name in TABLES:
        assert (tmp_path / "f" / name).read_text() == golden(name), name
    sam_dir = os.path.join(CASE, "sam")
    for name in sorted(os.listdir(sam_dir)):
        assert (tmp_path / "f" / name).read_text() == open(os.path.join(sam_dir, name)).read(), name
    # and the same files as the DataFrame path, run.log included
    assert (src, trc, tru) == dataframe_path(args, files, SAMPLES, str(tmp_path / "d"), dev)
    same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))


def test_case1_without_spike_in(dev, tmp_path):
    files = [os.path.join(CASE, s + ".fastq.gz") for s in SAMPLES]
    args = case1_args(spikeIn=False)
    files_path(args, files, SAMPLES, str(tmp_path / "f"), dev)
    dataframe_path(args, files, SAMPLES, str(tmp_path / "d"), dev)
    same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))
    assert "spike-in" not in (tmp_path / "f" / "mapped.csv").read_text().splitlines()[0]


@pytest.mark.parametrize("name", DIGEST_CASES)
def test_digest_cases(dev, tmp_path, name):
    """The unannotated form on the table baking leaves is complete_set.csv; run_to_files writes baking's side files."""
    from mirge_b200 import digest as DG
    from mirge_b200 import outputs as O

    d, meta, args, files = load_digest_case(name)
    names = meta["samples"]
    base = tmp_path / "b"
    base.mkdir()
    df, src, trc, tru, table = DG.baking(args, files, names, str(base), device=dev, batch_bytes=70_000, keep_table=True)
    order = df.attrs["_mirge_b200_keys"].order
    counts = torch.zeros((len(names), table.n_keys), dtype=torch.int32, device=dev.tdev)
    if len(order):
        counts[:, torch.from_numpy(order).to(dev.tdev)] = torch.from_numpy(df[names].to_numpy().T.astype(np.int32)).to(dev.tdev)
    rows = torch.from_numpy(order).to(dev.tdev)
    O.write_table_csv(tmp_path / "complete_set.csv", dev, table, rows, counts, names, slice_bytes=2048)
    assert (tmp_path / "complete_set.csv").read_text() == open(os.path.join(d, "complete_set.csv")).read()
    # run_to_files with the annotation libraries of ref_case1: the side files are baking's
    args.libraries_path, args.organism_name = os.path.join(CASE, "lib"), ORG
    got = files_path(args, files, names, str(tmp_path / "f"), dev, batch_bytes=70_000)
    assert got == (src, trc, tru)
    side = sorted(f for f in os.listdir(base) if f.endswith((".fa", "_umiCounts.csv")))
    assert side == sorted(f for f in os.listdir(tmp_path / "f") if f.endswith((".fa", "_umiCounts.csv")))
    for f in side:
        assert same_side_file(str(tmp_path / "f"), str(base), f), f
    dataframe_path(args, files, names, str(tmp_path / "d"), dev, batch_bytes=70_000)
    same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))


def quoted_libs(rng):
    """make_sam_libs with reference names that need CSV quoting or are not ASCII."""
    libs = make_sam_libs(rng, scale=0.2)
    odd = ['mir,1', 'say"x"', "café", 'a,"b"', "µRNA"]
    for k in ("mirna", "hairpin", "mature_trna", "snorna", "spike-in"):
        names, seqs = libs[k]
        libs[k] = ([odd[i % len(odd)] + "_" + n if i % 3 == 0 else n for i, n in enumerate(names)], seqs)
    return libs


def odd_sample(path, rng, libs, n=600):
    """Reads whose inserts carry ',', '"' and latin-1 bytes >= 0x80 (the digest keeps any byte as an exception)."""
    from tests.sam_cases import insert

    recs = []
    for k in range(n):
        s = list(insert(rng, libs))
        for _ in range(int(rng.integers(0, 3))):
            s[int(rng.integers(len(s)))] = str(rng.choice([",", '"', "\xe9", "\xff", "N"]))
        s = ("".join(s) + ILL + "ACGTAC")[:70]
        recs.append(b"@o%d\n%s\n+\n%s\n" % (k, s.encode("latin-1"), b"I" * len(s)))
    with open(path, "wb") as fh:
        fh.write(b"".join(recs))


@pytest.mark.parametrize("slice_bytes", [1, 3000])
def test_synthetic_many_samples_quoting_and_slices(dev, tmp_path, slice_bytes):
    rng = np.random.default_rng(71)
    libs = quoted_libs(rng)
    write_lib_dir(str(tmp_path / "lib"), libs)
    files, names = write_samples(str(tmp_path), libs, n_samples=3, reads=1500)
    odd_sample(str(tmp_path / "odd.fastq"), rng, libs)
    files, names = files + [str(tmp_path / "odd.fastq")], names + ['odd,"name"']
    args = make_args(libraries_path=str(tmp_path / "lib"), spikeIn=True, bam_out=True, tRNA_frag=True, tcf_out=True)
    files_path(args, files, names, str(tmp_path / "f"), dev, ref_db="miRBase", batch_bytes=60_000, slice_bytes=slice_bytes)
    dataframe_path(args, files, names, str(tmp_path / "d"), dev, ref_db="miRBase", batch_bytes=60_000)
    out = same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))
    assert "miRge3_tRNA.sam" in out and "s0.trim.collapse.fa" in out
    mapped = (tmp_path / "f" / "mapped.csv").read_bytes()
    body = mapped.split(b"\n", 1)[1] + (tmp_path / "f" / "unmapped.csv").read_bytes().split(b"\n", 1)[1]
    assert b'"odd,""name"""' in mapped.split(b"\n", 1)[0]
    assert re.search(rb',"[^"\n]*(,|"")', body)  # a quoted reference name
    assert b"\xc3\xa9" in body and b'""' in body  # keys with latin-1 bytes and with '"'


def test_empty_table_gives_the_header_only(dev, tmp_path):
    rng = np.random.default_rng(5)
    libs = make_sam_libs(rng, scale=0.1)
    write_lib_dir(str(tmp_path / "lib"), libs)
    with open(tmp_path / "short.fastq", "w") as fh:  # every read is shorter than the length filter's 16 nt
        fh.write("".join("@r%d\n%s\n+\n%s\n" % (k, "ACGTACGTAC", "I" * 10) for k in range(200)))
    args = make_args(libraries_path=str(tmp_path / "lib"))
    files_path(args, [str(tmp_path / "short.fastq")], ["s"], str(tmp_path / "f"), dev, ref_db="miRBase")
    dataframe_path(args, [str(tmp_path / "short.fastq")], ["s"], str(tmp_path / "d"), dev, ref_db="miRBase")
    same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))
    assert len((tmp_path / "f" / "mapped.csv").read_text().splitlines()) == 1
    assert len((tmp_path / "f" / "unmapped.csv").read_text().splitlines()) == 1


def test_table_above_one_million_rows(dev, tmp_path):
    """> 1 M rows: bwtAlign builds its annotation columns on the device (_fill_rounds_device) and the DataFrame index
    is Arrow-backed; run_to_files writes the same bytes in many slices."""
    from mirge_b200 import synth

    slibs = synth.make_libraries(scale=0.05, mrna_count=500)
    libs = {k: (list(v[0]), [s.decode() for s in v[1]]) for k, v in slibs.fasta_dict().items()}
    write_lib_dir(str(tmp_path / "lib"), libs)
    gen = synth.ReadGenerator(slibs, synth.CONFIGS[1], "cpu")
    rng = np.random.default_rng(9)
    names = ["lib_reads", "random_reads"]
    with open(tmp_path / "a.fastq", "wb") as fh:
        fh.write(gen.fastq(300_000).numpy().tobytes())
    n = 1_100_000  # random inserts of 18-34 nt: nearly all unique
    L = rng.integers(18, 35, size=n)
    codes = rng.integers(0, 4, size=(n, 34))
    seqs = np.frombuffer(b"ACGT", dtype=np.uint8)[codes]
    with open(tmp_path / "b.fastq", "wb") as fh:
        out = []
        for k in range(n):
            s = seqs[k, : L[k]].tobytes() + ILL.encode()[:16]
            out.append(b"@x%d\n%s\n+\n%s\n" % (k, s, b"I" * len(s)))
        fh.write(b"".join(out))
    files = [str(tmp_path / "a.fastq"), str(tmp_path / "b.fastq")]
    args = make_args(libraries_path=str(tmp_path / "lib"), spikeIn=True)
    files_path(args, files, names, str(tmp_path / "f"), dev, ref_db="miRBase", batch_bytes=32 << 20, slice_bytes=1 << 20)
    dataframe_path(args, files, names, str(tmp_path / "d"), dev, ref_db="miRBase", batch_bytes=32 << 20)
    same_outputs(str(tmp_path / "f"), str(tmp_path / "d"))
    rows = sum(1 for _ in open(tmp_path / "f" / "mapped.csv", "rb")) + sum(1 for _ in open(tmp_path / "f" / "unmapped.csv", "rb")) - 2
    assert rows > 1_000_000


@pytest.mark.parametrize("n_samples", [1, 40, 300])
def test_wide_rows_and_partial_ctas(dev, tmp_path, n_samples):
    """Rows of 1, 40 and 300 sample counts (up to 3 kB a row), formatted in one slice, in slices of a few rows and one
    row at a time."""
    import pandas as pd

    from mirge_b200 import digest as DG
    from mirge_b200 import outputs as O

    files = [os.path.join(CASE, s + ".fastq.gz") for s in SAMPLES]
    df, *_, table = DG.baking(case1_args(), files, SAMPLES, str(tmp_path), device=dev, keep_table=True)
    order = df.attrs["_mirge_b200_keys"].order
    rng = np.random.default_rng(n_samples)
    names = ["c%d" % j for j in range(n_samples)]
    cnt = rng.choice([0, 1, 7, 123456, 2**32 - 1], size=(n_samples, table.n_keys)).astype(np.uint32)
    frame = df[["annotFlag"] + DG.INITIAL_FLAGS].copy()
    for j, nm in enumerate(names):
        frame[nm] = cnt[j][order].astype(np.int64)
    exp = tmp_path / "exp.csv"
    pd.DataFrame(frame).to_csv(exp)
    counts = torch.from_numpy(cnt.view(np.int32)).to(dev.tdev)
    rows = torch.from_numpy(order).to(dev.tdev)
    for k, sb in enumerate((1 << 20, 5000, 1)):
        got = tmp_path / ("got%d.csv" % k)
        O.write_table_csv(got, dev, table, rows, counts, names, slice_bytes=sb)
        assert got.read_bytes() == exp.read_bytes(), sb
