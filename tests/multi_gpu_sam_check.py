"""Run under torchrun (one rank per GPU, one rank or more): baking_sharded + bwtAlign_sharded with -bam -trf write the
per-round SAM files from the owners' records, and every file must be byte-identical to the one the single-process
baking + bwtAlign writes on the same inputs (and the returned tables equal).  Argument ``umi``: reads with 4-base UMI
flanks and -udd.  The inputs include a sample of one repeated read, whose sequences all have one owner.  Used by
tests/test_gpu_sam.py; exits non-zero on any difference."""
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


def main():
    import shutil
    import tempfile

    from tests.sam_cases import make_sam_libs, write_samples
    from tests.test_gpu_annotate import write_lib_dir
    from tests.util import make_args

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = D.Device(local)
    umi = len(sys.argv) > 1 and sys.argv[1] == "umi"
    box = [tempfile.mkdtemp(prefix="mirge_sam_") if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    tmp = box[0]
    sharded, single = os.path.join(tmp, "sharded"), os.path.join(tmp, "single")
    if rank == 0:
        libs = make_sam_libs(np.random.default_rng(7), scale=0.3)
        write_lib_dir(os.path.join(tmp, "lib"), libs)
        files, names = write_samples(tmp, libs, n_samples=4, reads=2000, umi=umi)
        os.makedirs(sharded)
        os.makedirs(single)
    else:
        files = names = None
    box = [(files, names)]
    dist.broadcast_object_list(box, 0)
    files, names = box[0]
    args = make_args(libraries_path=os.path.join(tmp, "lib"), spikeIn=True, uniq_mol_ids="4,4" if umi else None, umiDedup=umi,
                     bam_out=True, tRNA_frag=True)
    df, *_ = MD.baking_sharded(args, files, names, sharded, device=dev, batch_bytes=150_000)
    out = MD.bwtAlign_sharded(args, df, sharded, "miRBase")
    dist.barrier()
    ok = True
    if rank == 0:
        df1, *_ = DG.baking(args, files, names, single, device=dev, batch_bytes=150_000)
        out1 = MA.bwtAlign(args, df1, single, "miRBase", device=dev)
        ok = out.equals(out1)
        sams = lambda d: sorted(f for f in os.listdir(d) if f.endswith(".sam"))
        ok = ok and sams(sharded) == sams(single) and "miRge3_tRNA.sam" in sams(single)
        n_bytes = 0
        for f in sams(single):
            a, b = open(os.path.join(sharded, f), "rb").read(), open(os.path.join(single, f), "rb").read()
            n_bytes += len(b)
            if a != b:
                ok = False
                print("differs:", f, len(a), len(b))
        print("sharded SAM files: world=%d umi=%s rows=%d files=%s bytes=%d ok=%s"
              % (world, umi, len(out1), sams(single), n_bytes, ok))
        shutil.rmtree(tmp, ignore_errors=True)
    flag = torch.tensor([1 if ok else 0], device=dev.tdev)
    dist.broadcast(flag, 0)
    dist.destroy_process_group()
    sys.exit(0 if int(flag.item()) == 1 else 1)


if __name__ == "__main__":
    main()
