"""Wall-clock cost of a run's output files: the DataFrame path against outputs.run_to_files, on a bench-size table.

One sample of a bench.py configuration (default C2: 50 M reads, mRNA 100 k entries, the bench's seeded libraries and
reads) is written to a FASTQ file; then, alternating, three times each (after one untimed pass of each):
  (a) baking + bwtAlign + report.write_tables + report.annotation_report
  (b) outputs.run_to_files
each timed from the call to the last file closed, with the output directory on /dev/shm.  Prints one JSON line: the
times, the CUDA-event time of the row-formatting kernel (both launches, all slices), the rows and bytes of mapped.csv
+ unmapped.csv, whether the two output sets are identical (run.log up to its timings), and the card's name and power
limit read in the same process.  Beside them, in the same process: the device-to-host copy of as many bytes as the
two CSV files hold, in 64 MB pieces into two pinned buffers as write_table_csv copies them (CUDA events), and the
host's write of those bytes from pinned memory to a file in the output directory (wall clock).

    python profiles/files_time.py [--tree DIR] [--reads N] [--reps R] [--out DIR]

``--tree`` imports the package from another checkout (e.g. the parent commit, built with its own
__graft_entry__.build()), so the formatting kernels of two versions can be compared on the same box."""
import argparse
import dataclasses
import json
import os
import re
import shutil
import sys
import tempfile
import time

sys.dont_write_bytecode = True
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)


def same_files(a, b):
    fa, fb = sorted(os.listdir(a)), sorted(os.listdir(b))
    if fa != fb:
        return False
    for f in fa:
        pa, pb = os.path.join(a, f), os.path.join(b, f)
        if f == "run.log":
            strip = lambda p: re.sub(r"in [0-9.e+-]+ second", "in T second", open(p).read())
            if strip(pa) != strip(pb):
                return False
            continue
        if os.path.getsize(pa) != os.path.getsize(pb):
            return False
        with open(pa, "rb") as x, open(pb, "rb") as y:
            for bx in iter(lambda: x.read(1 << 26), b""):
                if bx != y.read(1 << 26):
                    return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", type=int, default=2, choices=(1, 2))
    ap.add_argument("--reads", type=int, default=0, help="reads (default: the config's, 1 M for C1 and 50 M for C2)")
    ap.add_argument("--reps", type=int, default=3, help="timed passes of each variant (after one untimed pass)")
    ap.add_argument("--out", default="/dev/shm" if os.path.isdir("/dev/shm") else None, help="where the output directories go")
    ap.add_argument("--tree", default=os.path.dirname(HERE), help="checkout whose mirge_b200 is timed")
    a = ap.parse_args()
    tree = os.path.abspath(a.tree)
    sys.path.insert(0, tree)
    import torch

    import mirge_b200  # noqa: F401
    from mirge_b200 import device as D
    from mirge_b200 import digest as DG
    from mirge_b200 import libraries as LB
    from mirge_b200 import manifoldAlign as MA
    from mirge_b200 import outputs as O
    from mirge_b200 import report as RP
    from mirge_b200 import synth
    from sam_time import card
    from tests.util import make_args

    reads = a.reads or (1_000_000 if a.config == 1 else 50_000_000)
    mrna = 5_000 if a.config == 1 else 100_000
    dev = D.Device(0)
    libs = synth.make_libraries(mrna_count=mrna)
    lset = LB.LibrarySet.from_fasta_dict(dev, libs.fasta_dict())
    gen = synth.ReadGenerator(libs, dataclasses.replace(synth.CONFIGS[a.config], sample_seed=0), dev.tdev)
    gen.gen.manual_seed(2000 + a.config)
    fq = gen.fastq(reads, first_index=0)
    tmp = tempfile.mkdtemp(prefix="mirge_files_time_")
    out_root = tempfile.mkdtemp(prefix="mirge_files_out_", dir=a.out)
    try:
        path = os.path.join(tmp, "sample.fastq")
        with open(path, "wb") as fh:
            for lo in range(0, int(fq.numel()), 1 << 30):
                fh.write(fq[lo : lo + (1 << 30)].cpu().numpy().tobytes())
        del fq
        kw = dict(quiet=True, threads=os.cpu_count() or 1, libraries_path=tmp, organism_name="synth")
        if a.config == 2:
            kw.update(nextseq_trim=20, quality_cutoff="20")
        args = make_args(**kw)

        def dataframe(work):
            df, src, trc, tru = DG.baking(args, [path], ["sample"], work, device=dev)
            out = MA.bwtAlign(args, df, work, "miRBase", libraries=lset, device=dev)
            RP.write_tables(out, work)
            RP.annotation_report(args, work, "miRBase", ["sample"], out, src, trc, tru, libraries=lset, device=dev)

        def files(work):
            O.run_to_files(args, [path], ["sample"], work, "miRBase", device=dev, libraries=lset)

        variants = {"dataframe": dataframe, "run_to_files": files}
        times = {k: [] for k in variants}
        kernel_ms, identical, rows, nbytes = [], True, 0, 0
        for rep in range(a.reps + 1):
            dirs = {}
            for name, fn in variants.items():
                work = dirs[name] = os.path.join(out_root, "%s_%d" % (name, rep))
                os.makedirs(work)
                dev.timing = name == "run_to_files"
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                fn(work)
                torch.cuda.synchronize()
                t1 = time.perf_counter()
                if dev.timing:
                    tot = dev.timer_totals()
                    if rep:
                        kernel_ms.append(round(tot.get("csv_format", (0, 0.0))[1], 2))
                dev.timing = False
                if rep:
                    times[name].append(round(t1 - t0, 3))
            identical &= same_files(dirs["dataframe"], dirs["run_to_files"])
            nbytes, rows = 0, 0
            for f in ("mapped.csv", "unmapped.csv"):
                p = os.path.join(dirs["run_to_files"], f)
                nbytes += os.path.getsize(p)
                with open(p, "rb") as fh:
                    rows += sum(block.count(b"\n") for block in iter(lambda: fh.read(1 << 26), b"")) - 1
            for d in dirs.values():
                shutil.rmtree(d, ignore_errors=True)
        # what the text costs past the kernel: the copy to pinned host memory and the write to the output directory
        piece = 64 << 20
        text_d = torch.empty(nbytes, dtype=torch.uint8, device=dev.tdev)
        host = [torch.empty(piece, dtype=torch.uint8).pin_memory() for _ in range(2)]
        d2h_ms, write_s = [], []
        for rep in range(a.reps + 1):
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for k, lo in enumerate(range(0, nbytes, piece)):
                hi = min(lo + piece, nbytes)
                host[k % 2][: hi - lo].copy_(text_d[lo:hi], non_blocking=True)
            ev1.record()
            torch.cuda.synchronize()
            path_w = os.path.join(out_root, "write_probe")
            t0 = time.perf_counter()
            with open(path_w, "wb") as fh:
                for lo in range(0, nbytes, piece):
                    fh.write(memoryview(host[0].numpy())[: min(piece, nbytes - lo)])
            t1 = time.perf_counter()
            os.remove(path_w)
            if rep:
                d2h_ms.append(round(ev0.elapsed_time(ev1), 2))
                write_s.append(round(t1 - t0, 3))
        del text_d
        name, power = card()
        print(json.dumps({"tree": tree, "config": a.config, "reads": reads, "rows": rows, "csv_bytes": nbytes,
                          "dataframe_path_s": times["dataframe"], "run_to_files_s": times["run_to_files"],
                          "csv_format_kernel_ms": kernel_ms, "d2h_copy_ms": d2h_ms, "host_write_s": write_s, "identical": bool(identical), "out_dir": a.out or "tmp",
                          "gpu": name, "power_limit": power}), flush=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
        shutil.rmtree(out_root, ignore_errors=True)


if __name__ == "__main__":
    main()
