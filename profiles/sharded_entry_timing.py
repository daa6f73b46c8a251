"""Time the multi-GPU entry points, distributed.baking_sharded + bwtAlign_sharded, on a seeded synthetic cohort.

Run under torchrun with one process per GPU, e.g.

    torchrun --nproc-per-node 4 profiles/sharded_entry_timing.py --samples 8 --reads 20000000 --gzip 1 --dir /dev/shm/cohort

Rank 0 writes the cohort once (C4-like reads, synth.CONFIGS[4] with a per-sample seed): ``--samples`` plain FASTQ files
plus ``--gzip`` gzip files, into ``--dir`` (RAM-backed, so that reading is not the disk's speed).  Each of ``--repeat``
runs times both entry points with the host clock around work that ends in a device synchronise and a barrier.  Rank 0
prints one JSON line per run: seconds per stage, world, GPU name and power limit, and a hash of the returned DataFrame.

``--impl ROOT`` imports the package from another checkout (its library built there), so that two versions can be timed
alternately in one job: ``--impl . --impl /path/to/older`` runs them in turn, ``--repeat`` times each."""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(HERE)


def gpu_info(index):
    """(name, power limit) of the GPU, read in the same job as the measurement"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return name, limit
    except Exception:
        import torch

        return torch.cuda.get_device_name(index), "unknown"


def write_cohort(d, n_samples, n_gzip, reads):
    import gzip

    from mirge_b200 import synth

    os.makedirs(d, exist_ok=True)
    libs = synth.make_libraries()
    files = []
    for i in range(n_samples + n_gzip):
        gz = i >= n_samples
        path = os.path.join(d, "c4_%02d.fastq%s" % (i, ".gz" if gz else ""))
        files.append(path)
        if os.path.exists(path):
            continue
        rc = synth.ReadConfig(4, 50, sample_seed=i + 1)
        gen = synth.ReadGenerator(libs, rc, "cpu")
        tmp = path + ".part"
        with (gzip.open(tmp, "wb", compresslevel=1) if gz else open(tmp, "wb")) as fh:
            step = 2_000_000
            for a in range(0, reads, step):
                fh.write(gen.fastq(min(step, reads - a)).numpy().tobytes())
        os.replace(tmp, path)
    return files, libs


def load_impl(root):
    """the package of checkout ``root`` (fresh import)"""
    for name in [m for m in sys.modules if m == "mirge_b200" or m.startswith("mirge_b200.")]:
        del sys.modules[name]
    sys.path.insert(0, os.path.abspath(root))
    try:
        importlib.import_module("mirge_b200")
        return {k: importlib.import_module("mirge_b200." + k) for k in ("device", "distributed", "libraries")}
    finally:
        sys.path.pop(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=8)
    ap.add_argument("--gzip", type=int, default=1)
    ap.add_argument("--reads", type=int, default=20_000_000)
    ap.add_argument("--dir", default="/dev/shm/mirge_cohort")
    ap.add_argument("--repeat", type=int, default=2)
    ap.add_argument("--impl", action="append", default=None)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file (rank 0)")
    a = ap.parse_args()

    import torch
    import torch.distributed as dist

    sys.path.insert(0, REPO)
    from tests.util import make_args

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    impls = a.impl or [REPO]
    if rank == 0:
        load_impl(impls[0])
        files, _ = write_cohort(a.dir, a.samples, a.gzip, a.reads)
    box = [files if rank == 0 else None]
    dist.broadcast_object_list(box, 0)
    files = box[0]
    names = [os.path.basename(f).split(".")[0] for f in files]
    name, limit = gpu_info(local)
    work = os.path.join(a.dir, "work_%d" % rank)
    os.makedirs(work, exist_ok=True)
    for rep in range(a.repeat):
        for root in impls:
            m = load_impl(root)
            D, MD, LB = m["device"], m["distributed"], m["libraries"]
            from mirge_b200 import synth

            dev = D.Device(local)
            libs = LB.LibrarySet.from_fasta_dict(dev, synth.make_libraries().fasta_dict())
            args = make_args(threads=max(1, (os.cpu_count() or 8) // world))
            dist.barrier()
            t0 = time.perf_counter()
            df, src, trc, tru = MD.baking_sharded(args, files, names, work, device=dev)
            torch.cuda.synchronize()
            dist.barrier()
            t1 = time.perf_counter()
            out = MD.bwtAlign_sharded(args, df, work, "miRBase", libraries=libs)
            torch.cuda.synchronize()
            dist.barrier()
            t2 = time.perf_counter()
            if rank == 0:
                digest = hashlib.sha256(out.to_csv().encode()).hexdigest()[:16]
                rec = {"impl": os.path.abspath(root), "run": rep, "world": world, "gpu": name, "power_limit": limit,
                       "samples": len(files), "gzip_samples": a.gzip, "reads_per_sample": a.reads,
                       "baking_sharded_s": round(t1 - t0, 3), "bwtAlign_sharded_s": round(t2 - t1, 3),
                       "rows": int(len(out)), "records": int(sum(src.values())), "frame_sha256": digest}
                line = json.dumps(rec)
                print(line, flush=True)
                if a.out:
                    with open(a.out, "a") as fh:
                        fh.write(line + "\n")
            del df, out, libs, dev
            torch.cuda.empty_cache()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
