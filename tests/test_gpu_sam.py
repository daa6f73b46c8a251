"""The per-round SAM files of -bam / -trf formatted on the GPU (mirge_sam_format, csrc/sam_format.cuh):
(a) every record of every annotated sequence of a synthetic table against pyoracle.sam_line, with tRNA libraries whose
duplicates and near duplicates give several best-stratum hits per sequence in rounds 2 and 3;
(b) bwtAlign with -bam -trf on a frame straight from baking (packed keys still on the device) and on the same frame
read back from CSV (keys packed from the index strings): the same files, equal to the oracle's, and the same table as
without the flags;
(c) baking_sharded + bwtAlign_sharded under torch.distributed.run (one rank; two where two GPUs exist): the files are
byte-identical to the single-process ones (tests/multi_gpu_sam_check.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import pyoracle as po
from tests.sam_cases import expected_sam_files, insert, make_sam_libs, round_hits, write_samples
from tests.test_gpu_annotate import make_queries, write_lib_dir
from tests.util import make_args

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SAM_NAMES = ["miRge3_miRNA.sam", "miRge3_hairpin_miRNA.sam", "miRge3_tRNA.sam", "miRge3_pre_tRNA.sam", "miRge3_snorna.sam",
             "miRge3_rrna.sam", "miRge3_ncrna_others.sam", "miRge3_mrna.sam"]


@pytest.fixture(scope="module")
def dev():
    from mirge_b200 import device as D

    return D.Device(0)


def test_device_records_equal_the_oracle(dev):
    from mirge_b200 import libraries as LB
    from mirge_b200 import manifoldAlign as MA

    rng = np.random.default_rng(31)
    libs = make_sam_libs(rng, scale=0.2)
    seqs = sorted(set(make_queries(rng, libs, 1500)) | {insert(rng, libs) for _ in range(1500)})
    ls = LB.LibrarySet.from_fasta_dict(dev, {k: (n, [s.encode() for s in v]) for k, (n, v) in libs.items()})
    ks = MA.KeySet.from_strings(dev, seqs)
    annot, hit = MA.annotate_keys(dev, ls, ks, True)
    annot_h = annot.cpu().numpy()
    pols = LB.round_policies()
    n_rec, multi = 0, 0
    for rnd in range(10):
        ids = np.nonzero(annot_h == rnd)[0]
        assert ids.size, rnd
        lib = ls[LB.ROUND_LIBS[rnd]]
        names, refs = libs[LB.ROUND_LIBS[rnd]]
        plib = po.Library(list(names), [r.upper() for r in refs])
        rec_ids, rec_hits = MA.round_sam_pairs(dev, lib, pols[rnd], ks, ids, hit)
        words = rec_hits.cpu().numpy().view(np.uint64)
        # small slices: the fill launch runs many times per round
        parts = list(MA.sam_records(dev, lib, pols[rnd], ks, rec_ids, rec_hits, slice_bytes=4096))
        assert len(parts) > 1 or rec_ids.size < 20
        data = b"".join(p.tobytes() for p, _ in parts)
        lens = np.concatenate([n for _, n in parts])
        assert lens.size == rec_ids.size and int(lens.sum()) == len(data)
        recs = data.split(b"\n")[:-1]
        assert len(recs) == rec_ids.size
        at = 0
        for i in ids.tolist():
            s = seqs[i]
            q = MA.round_query_text(s, pols[rnd])
            exp = round_hits(q, plib, rnd)
            got = words[at : at + len(exp)].tolist()
            assert got == exp and (rec_ids[at : at + len(exp)] == i).all(), (rnd, s, got, exp)
            multi += len(exp) > 1
            for w in exp:
                r, off = (w >> 28) & 0xFFFFFFF, w & 0xFFFFFFF
                line = po.sam_line(s, q, plib.names[r], plib.seqs[r], off, po.ROUND_POLICIES[rnd])
                assert recs[at].decode("latin-1") == line, (rnd, recs[at], line)
                at += 1
        n_rec += at
    assert multi > 20 and n_rec > 1000, (multi, n_rec)


def _frame_from_csv(df, path):
    """The table the way a caller that stored it would hand it back: no device keys, index from the CSV text."""
    import pandas as pd

    df.to_csv(path)
    back = pd.read_csv(path, index_col=0, keep_default_na=False)
    for c in back.columns:
        if back[c].dtype != np.int64:
            back[c] = back[c].astype(object)
    return back


def test_bwtalign_files_on_device_keys_and_strings(dev, tmp_path, monkeypatch):
    from mirge_b200 import digest as DG
    from mirge_b200 import manifoldAlign as MA

    rng = np.random.default_rng(32)
    libs = make_sam_libs(rng, scale=0.2)
    write_lib_dir(str(tmp_path / "lib"), libs)
    files, names = write_samples(str(tmp_path), libs)
    plain = make_args(libraries_path=str(tmp_path / "lib"), spikeIn=True)
    flags = make_args(libraries_path=str(tmp_path / "lib"), spikeIn=True, bam_out=True, tRNA_frag=True)
    runs = {}
    for name, args in (("plain", plain), ("device", flags), ("strings", flags)):
        work = tmp_path / name
        work.mkdir()
        df, *_ = DG.baking(args, files, names, str(work), device=dev, batch_bytes=60_000)
        if name == "strings":
            df = _frame_from_csv(df, str(tmp_path / "frame.csv"))
        with monkeypatch.context() as m:
            if name == "device":  # the packed keys of the table must serve: no index string is packed again
                m.setattr(MA.KeySet, "from_strings", classmethod(lambda *a, **k: (_ for _ in ()).throw(AssertionError("from_strings"))))
            runs[name] = MA.bwtAlign(args, df, str(work), "miRBase", device=dev)
    assert runs["device"].equals(runs["plain"])
    assert runs["strings"].astype(str).equals(runs["plain"].astype(str))
    exp = expected_sam_files(runs["plain"], libs, True, True, True)
    assert set(exp) <= set(SAM_NAMES)
    assert "miRge3_tRNA.sam" in exp and "miRge3_pre_tRNA.sam" in exp and "miRge3_miRNA.sam" in exp
    for name in ("device", "strings"):
        written = sorted(f for f in os.listdir(tmp_path / name) if f.endswith(".sam"))
        assert written == sorted(exp), (name, written)
        for f, text in exp.items():
            assert (tmp_path / name / f).read_bytes() == text.encode(), (name, f)
    assert not any(f.endswith(".sam") for f in os.listdir(tmp_path / "plain"))


@pytest.mark.parametrize("world,umi", [(1, False), (1, True), (2, False), (2, True)])
def test_sharded_entry_points_write_the_single_process_files(world, umi):
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29640 + 2 * world + int(umi)), os.path.join(ROOT, "tests", "multi_gpu_sam_check.py")] + (["umi"] if umi else [])
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "ok=True" in p.stdout
