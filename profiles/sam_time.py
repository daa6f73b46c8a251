"""Wall-clock cost of the per-round SAM files (-bam / -trf) in bwtAlign on a bench-size table.

One sample of a bench.py configuration (default C2: 50 M reads, mRNA 100 k entries, the bench's seeded libraries and
reads) goes through baking(); bwtAlign then runs on the fresh frame without and with -bam -trf, each timed from the
call to its return after a device synchronise.  Prints one JSON line: the two times, the SAM records and bytes
written, and the card's name and power limit read in the same process.

    python profiles/sam_time.py [--tree DIR] [--reads N] [--reps R]

``--tree`` imports the package from another checkout (e.g. the parent commit, built with its own
__graft_entry__.build()), so two versions can be compared in one job, alternating."""
import argparse
import dataclasses
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))


def card():
    import torch

    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tree", default=os.path.dirname(HERE), help="checkout whose mirge_b200 is timed")
    ap.add_argument("--config", type=int, default=2, choices=(1, 2))
    ap.add_argument("--reads", type=int, default=0, help="reads (default: the config's, 1 M for C1 and 50 M for C2)")
    ap.add_argument("--mrna", type=int, default=0, help="mRNA library entries (default: the config's)")
    ap.add_argument("--reps", type=int, default=2, help="timed passes of each variant (after one untimed pass)")
    a = ap.parse_args()
    tree = os.path.abspath(a.tree)
    sys.path.insert(0, tree)
    import numpy as np
    import torch

    import mirge_b200  # noqa: F401
    from mirge_b200 import device as D
    from mirge_b200 import digest as DG
    from mirge_b200 import libraries as LB
    from mirge_b200 import manifoldAlign as MA
    from mirge_b200 import synth
    from tests.util import make_args

    reads = a.reads or (1_000_000 if a.config == 1 else 50_000_000)
    mrna = a.mrna or (5_000 if a.config == 1 else 100_000)
    dev = D.Device(0)
    libs = synth.make_libraries(mrna_count=mrna)
    lset = LB.LibrarySet.from_fasta_dict(dev, libs.fasta_dict())
    # the bench's sample 0 of the configuration (bench.py sample_fastq)
    gen = synth.ReadGenerator(libs, dataclasses.replace(synth.CONFIGS[a.config], sample_seed=0), dev.tdev)
    gen.gen.manual_seed(2000 + a.config)
    fq = gen.fastq(reads, first_index=0)
    tmp = tempfile.mkdtemp(prefix="mirge_sam_time_")
    try:
        path = os.path.join(tmp, "sample.fastq")
        with open(path, "wb") as fh:
            for lo in range(0, int(fq.numel()), 1 << 30):
                fh.write(fq[lo : lo + (1 << 30)].cpu().numpy().tobytes())
        del fq
        kw = dict(quiet=True, threads=os.cpu_count() or 1)
        if a.config == 2:
            kw.update(nextseq_trim=20, quality_cutoff="20")
        variants = {"plain": make_args(**kw), "bam_trf": make_args(bam_out=True, tRNA_frag=True, **kw)}
        times = {k: [] for k in variants}
        rows = records = sam_bytes = 0
        for rep in range(a.reps + 1):
            for name, args in variants.items():
                work = os.path.join(tmp, "%s_%d" % (name, rep))
                os.makedirs(work)
                df, *_ = DG.baking(args, [path], ["sample"], work, device=dev)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                out = MA.bwtAlign(args, df, work, "miRBase", libraries=lset, device=dev)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                if rep:
                    times[name].append(t1 - t0)
                rows = len(out)
                if name == "bam_trf":
                    sams = [os.path.join(work, f) for f in os.listdir(work) if f.endswith(".sam")]
                    sam_bytes = sum(os.path.getsize(f) for f in sams)
                    records = 0
                    for f in sams:
                        with open(f, "rb") as fh:
                            for block in iter(lambda: fh.read(1 << 26), b""):
                                records += block.count(b"\n")
                del df, out
                shutil.rmtree(work, ignore_errors=True)
        name, power = card()
        print(json.dumps({"tree": tree, "config": a.config, "reads": reads, "rows": rows,
                          "bwtAlign_s": [round(t, 3) for t in times["plain"]],
                          "bwtAlign_bam_trf_s": [round(t, 3) for t in times["bam_trf"]],
                          "sam_records": records, "sam_bytes": sam_bytes, "gpu": name, "power_limit": power}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == "__main__":
    main()
