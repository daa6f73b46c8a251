"""Run under torchrun (one rank per GPU, one rank or more): baking_sharded + bwtAlign_sharded, which digest every sample
on all ranks (plain files cut into record-aligned byte ranges, gzip files read by one rank, keys sent to their owners
before the collapse), against the single-process baking + bwtAlign on the same inputs.  The DataFrame must be equal,
the counters equal, the SAM files byte-identical and the -tcf / _umiCounts.csv rows equal as multisets.

Cases: ``plain`` (-tcf -bam -trf; plain samples, one of a single record, and a gzip sample), ``umi`` (-umi 4,4 -udd
-tcf -bam -trf), ``qiagen`` (--qiagenumi -umi 0,12 -udd -tcf).  Used by tests/test_gpu_split_samples.py; exits non-zero
on any difference."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mirge_b200  # noqa: E402,F401
from mirge_b200 import device as D  # noqa: E402
from mirge_b200 import digest as DG  # noqa: E402
from mirge_b200 import distributed as MD  # noqa: E402
from mirge_b200 import manifoldAlign as MA  # noqa: E402
from mirge_b200 import synth  # noqa: E402


def write_inputs(tmp, case):
    from tests.sam_cases import make_sam_libs, write_samples
    from tests.test_gpu_annotate import write_lib_dir

    libs = make_sam_libs(np.random.default_rng(7), scale=0.3)
    write_lib_dir(os.path.join(tmp, "lib"), libs)
    if case == "qiagen":
        files, names = [], []
        for i in range(3):
            rc = synth.ReadConfig(3, 75, adapter=synth.QIA_INNER, qiaseq=True, sample_seed=i)
            data = synth.ReadGenerator(synth.make_libraries(scale=0.05, mrna_count=100), rc, "cpu").fastq(3000 + 500 * i).numpy()
            files.append(os.path.join(tmp, "q%d.fastq" % i))
            names.append("q%d" % i)
            data.tofile(files[-1])
        return files, names
    # s1 is gzipped, the last sample repeats one read
    files, names = write_samples(tmp, libs, n_samples=4, reads=2500, umi=case == "umi")
    one = os.path.join(tmp, "tiny.fastq")  # fewer records than ranks: some ranks get an empty byte range
    with open(files[0], "rb") as fh:
        head = fh.read().split(b"\n")[:4]
    with open(one, "wb") as fh:
        fh.write(b"\n".join(head) + b"\n")
    return files[:2] + [one] + files[2:], names[:2] + ["tiny"] + names[2:]


def tcf_rows(d, names):
    """{sample: sorted [(count, sequence)]} of the <sample>.trim.collapse.fa files; counts must descend"""
    got = {}
    for n in names:
        lines = open(os.path.join(d, n + ".trim.collapse.fa")).read().split("\n")
        recs = [(int(h.rsplit("_", 1)[1]), s_) for h, s_ in zip(lines[0::2], lines[1::2]) if h]
        assert all(recs[i][0] >= recs[i + 1][0] for i in range(len(recs) - 1))
        assert [h for h in lines[0::2] if h] == [">seq%d_%d" % (i + 1, c) for i, (c, _) in enumerate(recs)]
        got[n] = sorted(recs)
    return got


def umi_rows(d, names):
    """{sample: (header, sorted rows)} of the <sample>_umiCounts.csv files"""
    got = {}
    for n in names:
        lines = open(os.path.join(d, n + "_umiCounts.csv")).read().split("\n")
        got[n] = (lines[0], sorted(lines[1:]))
    return got


def main():
    import shutil
    import tempfile

    from tests.util import make_args

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = D.Device(local)
    case = sys.argv[1]
    box = [tempfile.mkdtemp(prefix="mirge_split_") if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    tmp = box[0]
    sharded, single = os.path.join(tmp, "sharded"), os.path.join(tmp, "single")
    box = [write_inputs(tmp, case) if rank == 0 else None]
    if rank == 0:
        os.makedirs(sharded)
        os.makedirs(single)
    dist.broadcast_object_list(box, 0)
    files, names = box[0]
    kw = dict(libraries_path=os.path.join(tmp, "lib"), spikeIn=True, tcf_out=True)
    if case == "qiagen":
        kw.update(adapters=[("back", synth.QIA_INNER)], uniq_mol_ids="0,12", qiagenumi=True, umiDedup=True)
    else:
        kw.update(bam_out=True, tRNA_frag=True)
        if case == "umi":
            kw.update(uniq_mol_ids="4,4", umiDedup=True)
    args = make_args(**kw)
    df, src, trc, tru = MD.baking_sharded(args, files, names, sharded, device=dev, batch_bytes=150_000)
    out = MD.bwtAlign_sharded(args, df, sharded, "miRBase")
    dist.barrier()
    ok = True
    if rank == 0:
        df1, src1, trc1, tru1 = DG.baking(args, files, names, single, device=dev, batch_bytes=150_000)
        out1 = MA.bwtAlign(args, df1, single, "miRBase", device=dev)
        checks = {"frame": out.equals(out1) and list(out.columns) == list(out1.columns) and list(out.dtypes) == list(out1.dtypes),
                  "counters": (src, trc, tru) == (src1, trc1, tru1), "tcf": tcf_rows(sharded, names) == tcf_rows(single, names)}
        if kw.get("umiDedup"):
            checks["umiCounts"] = umi_rows(sharded, names) == umi_rows(single, names)
        sams = lambda d: sorted(f for f in os.listdir(d) if f.endswith(".sam"))
        checks["sam"] = sams(sharded) == sams(single)
        for f in sams(single):
            if open(os.path.join(sharded, f), "rb").read() != open(os.path.join(single, f), "rb").read():
                checks["sam"] = False
                print("differs:", f)
        ok = all(checks.values())
        print("split samples: world=%d case=%s rows=%d annotated=%d reads=%d checks=%s ok=%s"
              % (world, case, len(out1), int((out1.annotFlag == 1).sum()), sum(src1.values()), checks, ok))
        if not ok:
            print(src, src1, trc, trc1, tru, tru1, out.shape, out1.shape)
        shutil.rmtree(tmp, ignore_errors=True)
    flag = torch.tensor([1 if ok else 0], device=dev.tdev)
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
