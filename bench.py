#!/usr/bin/env python
"""bench.py -- throughput of the digest -> collapse -> annotate hot path on synthetic reads.

    python bench.py --gpus N --steps K --warmup W            (this repo's CUDA path)
    python bench.py --impl reference --gpus N --steps K ...   (CPU path: the oracle port, all host threads)
    python bench.py --gpus 1 ... --dump-outputs DIR           (also writes the last timed step's result table as .npy files,
                                                               for comparing two builds output for output)

Workload (BASELINE.json configs[1], SURVEY.md section 8d): 50 M-read single sample, L = 75, NextSeq poly-G
tails, ``-a illumina -nxt 20 -q 20``, all ordered libraries incl. a 100 000-entry mRNA library.  A step is
one whole pass of the hot path over that sample: tokenise -> trim -> collapse -> 9 annotation rounds.
``value``: inputs resident in HBM.  ``e2e``: the same pass fed from pinned HOST memory through the
streaming entry point (H2D of every input byte and D2H of the result table inside the timed region).
Multi-GPU (weak scaling): every rank trims its own 50 M-read shard; the keys of every batch are hash-
partitioned to their owner rank (all-to-all under the next batch's trim), owners collapse and annotate
their slice.  Multi-sample / UMI configurations collapse locally and exchange unique sequences per sample.
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the bench writes nothing into the tree it runs from (which may be read-only)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "M reads/s trim+collapse+annotate"
UNIT = "M reads/s"
# BASELINE.json configs (BASELINE.md section 3): reads per sample, samples per GPU, mRNA entries, spike-in round, label.
# C2 is the configuration the metric is quoted on and the default; C4 / C5 are per-GPU shares of the multi-GPU
# configurations (48 samples = 6 per GPU x 8, 1 B reads = 125 M per GPU x 8).
CONFIG_TABLE = {
    1: dict(reads=1_000_000, samples=1, mrna=5_000, spike=False,
            label="C1: 1M-read synthetic Illumina small-RNA sample, L=50, -a illumina (default -q 10), 9 rounds (mRNA 5k entries)"),
    2: dict(reads=50_000_000, samples=1, mrna=100_000, spike=False,
            label="C2: 50M-read single sample, L=75, -a illumina -nxt 20 -q 20, full ordered library annotation (mRNA 100k entries)"),
    3: dict(reads=100_000_000, samples=1, mrna=100_000, spike=False,
            label="C3: 100M-read QIAseq-style UMI library, L=75, -a AACTGTAGGCACCATCAAT --qiagenumi -umi 0,12 -udd, UMI-aware collapse"),
    4: dict(reads=20_000_000, samples=6, mrna=100_000, spike=False,
            label="C4 share: 6 samples x 20M reads per GPU (48 samples at 8 GPUs), L=50, -a illumina, per-sample counts"),
    5: dict(reads=125_000_000, samples=1, mrna=100_000, spike=True,
            label="C5 share: 125M reads per GPU (1B pooled at 8 GPUs), L=75, -a illumina -spk, 10 rounds incl. mRNA and spike-ins"),
}
CFG_ID = 2
WORKLOAD = CONFIG_TABLE[2]["label"]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIG_TABLE), help="BASELINE.json config (default 2: the metric's)")
    ap.add_argument("--reads", type=int, default=0, help="reads per sample and GPU (default: the config's)")
    ap.add_argument("--samples", type=int, default=0, help="samples per GPU (default: the config's)")
    ap.add_argument("--mrna", type=int, default=0, help="mRNA library entries (default: the config's)")
    ap.add_argument("--dropin", action="store_true",
                    help="also time baking(args, [file on /dev/shm]) + bwtAlign(args, df) -- the reference's entry points -- on one sample")
    ap.add_argument("--count-mode", default="head", choices=["head", "release"])
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="reads of the bounded CPU sample (0 = 12 M for the cpu_baseline leg, 4 M per step for --impl reference)")
    ap.add_argument("--batch-mb", type=int, default=2048)
    ap.add_argument("--e2e-batch-mb", type=int, default=256, help="piece size of the host-fed (e2e) pipeline")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--overlap-exchange", action="store_true", help="N > 1: per-batch exchange on a worker thread / side stream")
    ap.add_argument("--exchange-unique", action="store_true",
                    help="N > 1, single-sample configs: local collapse + exchange of the unique sequences instead of sharding before the collapse")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64 / float32, < 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    c = CONFIG_TABLE[a.config]
    a.reads = a.reads or c["reads"]
    a.samples = a.samples or c["samples"]
    a.mrna = a.mrna or c["mrna"]
    a.spike = c["spike"]
    a.workload = c["label"] if (a.reads, a.samples, a.mrna) == (c["reads"], c["samples"], c["mrna"]) else \
        c["label"] + " [reduced: %d reads x %d samples, mRNA %d]" % (a.reads, a.samples, a.mrna)
    return a


# ------------------------------------------------------------------------------------------------
# CPU arm (oracle port) -- cpu_baseline of the b200 line and the whole of --impl reference
# ------------------------------------------------------------------------------------------------


class CpuPath:
    """The reference's CPU path restated (oracle/mirge_oracle.c): cutadapt-semantics digest + dict collapse
    + the ordered rounds with an indexed bowtie-semantics search.  kind = "port": cutadapt / bowtie are not
    installable here, so the reference itself cannot be timed (DESIGN.md)."""

    def __init__(self, libs, cfg, threads):
        from mirge_b200 import params as P
        from mirge_b200.libraries import ROUND_LIBS, round_policies
        from oracle import coracle

        self.co = coracle
        self.threads = threads
        self.cfg = cfg
        self.cp = P.build_trim_params(cfg)
        self.pols = round_policies()
        self.round_libs = ROUND_LIBS
        self.index = {}
        lut = np.frombuffer(b"ACGTN", dtype=np.uint8)
        for key, L in libs.libs.items():
            self.index[key] = coracle.Index(lut[L.codes], L.off.astype(np.uint32))

    def step(self, fq: np.ndarray, spike=False):
        co = self.co
        n, tab = co.digest_collapse(fq, self.cp, nthreads=self.threads)
        umi = self.cfg.umi()
        if umi is not None:  # second level (digest.py:164-205), -udd
            tab = tab.umi_collapse(umi[0], umi[1], self.cfg.minimum_length, True)
        keys, off, cnt = tab.export()
        ar = np.full(len(cnt), 0xFF, dtype=np.uint8)
        hit = np.full(len(cnt), 0xFFFFFFFFFFFFFFFF, dtype=np.uint64)
        for rnd in range(10 if spike else 9):
            co.annotate_round_indexed(keys, off, self.index[self.round_libs[rnd]], self.pols[rnd], ar, hit, self.threads)
        return n, len(cnt), int((ar != 0xFF).sum())


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import mirge_b200  # noqa: F401
    from mirge_b200 import synth

    threads = host_threads()
    libs = synth.make_libraries(mrna_count=args.mrna)
    cfg = synth.trim_config_for(args.config, args.count_mode)
    cpu = CpuPath(libs, cfg, threads)
    gen = synth.ReadGenerator(libs, synth.CONFIGS[args.config], "cpu")
    sample = min(args.cpu_sample or 4_000_000, args.reads * args.samples)
    fq = gen.fastq(sample).numpy()
    for _ in range(args.warmup):
        cpu.step(fq, args.spike)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        n, nu, na = cpu.step(fq, args.spike)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    v = sample / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
        "config": {"workload": args.workload, "count_mode": args.count_mode, "reads_per_step": sample,
                   "note": "bounded sample of the workload per step; CPU only"},
        "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": threads, "kind": "port",
                         "sample": "%d reads of the workload per step (oracle port: cutadapt/bowtie not installable)" % sample},
        "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "50"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        for ln in self.f.read().splitlines():
            c = [x.strip() for x in ln.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}
        return out


def bind_to_gpu_numa_node(gpu_index):
    """Run this process on the CPUs next to its GPU (NVML's affinity mask) where the container's CPU set allows it, so
    that pinned host buffers are first touched on the GPU's own NUMA node and the copy threads stay there."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        near = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        pick = near & allowed
        if pick and pick != allowed:
            os.sched_setaffinity(0, pick)
        return sorted(pick)
    except Exception:
        return None


def single_stream_gzip(unit: bytes, reps: int, level: int = 6) -> bytes:
    """`reps` copies of `unit` as ONE gzip member holding ONE DEFLATE stream, at the cost of compressing the unit once:
    the unit's blocks end in a full flush (byte-aligned, dictionary reset), so they can be repeated verbatim; a final
    empty block, CRC-32 and ISIZE of the whole text close the member."""
    import struct
    import zlib

    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    body = c.compress(unit) + c.flush(zlib.Z_FULL_FLUSH)
    crc = 0
    for _ in range(reps):
        crc = zlib.crc32(unit, crc)
    last = zlib.compressobj(level, zlib.DEFLATED, -15).flush()  # BFINAL = 1, no data
    head = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\xff"
    return head + body * reps + last + struct.pack("<II", crc & 0xFFFFFFFF, (len(unit) * reps) & 0xFFFFFFFF)


def run_ingest_gz(fastq: np.ndarray, threads: int, target_mb: int = 512):
    """Host-side leg (no device work): the same synthetic FASTQ as a single-stream .fastq.gz -- what the reference's
    xopen(FQfile, "rb") meets in practice (digest.py:136) -- read through ingest.open_fastq: the chunk-parallel decoder
    (csrc/pinflate.c) on `threads` cores against the serial zlib reader, MB/s of FASTQ text delivered."""
    from mirge_b200 import ingest

    unit = fastq.tobytes()
    reps = max(1, (target_mb << 20) // max(len(unit), 1))
    tmpdir = tempfile.mkdtemp(prefix="mirge_gz_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    path = os.path.join(tmpdir, "sample.fastq.gz")
    try:
        blob = single_stream_gzip(unit, reps)
        with open(path, "wb") as f:
            f.write(blob)
        total = len(unit) * reps
        buf = bytearray(64 << 20)

        def read_all(th, parallel):
            os.environ["MIRGE_B200_PARALLEL_GZIP"] = "1" if parallel else "0"
            t0 = time.perf_counter()
            got = 0
            with ingest.open_fastq(path, threads=th) as r:
                while True:
                    k = r.readinto(buf)
                    if not k:
                        break
                    got += k
                    if not parallel and got >= (128 << 20):  # the serial reader is timed on the first 128 MB
                        break
            return got, time.perf_counter() - t0

        prev = os.environ.get("MIRGE_B200_PARALLEL_GZIP")
        try:
            read_all(threads, True)  # first pass: page faults of the decoder's buffers, thread start
            best = None
            for _ in range(3):
                got, dt = read_all(threads, True)
                if got != total:
                    raise RuntimeError("parallel gzip reader returned %d of %d bytes" % (got, total))
                best = dt if best is None else min(best, dt)
            g1, d1 = read_all(1, False)
        finally:
            if prev is None:
                os.environ.pop("MIRGE_B200_PARALLEL_GZIP", None)
            else:
                os.environ["MIRGE_B200_PARALLEL_GZIP"] = prev
        return {"value": round(total / best / 1e6, 1), "unit": "MB/s of FASTQ out of one .fastq.gz stream", "threads": threads,
                "serial_zlib_mb_s": round(g1 / d1 / 1e6, 1), "gz_mb": round(len(blob) / 1e6, 1), "fastq_mb": round(total / 1e6, 1),
                "ratio": round(total / len(blob), 2), "native_decoder": ingest.parallel_gzip_library() is not None,
                "note": "host cores only; best of 3 after a warm-up pass; through ingest.open_fastq (reader thread + decoder)"}
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)


def run_ingest_gz_guarded(fastq: np.ndarray, threads: int, timeout_s: int = 240):
    """run_ingest_gz in a process of its own with a time limit: the leg starts threads (decoder, reader) and is an extra --
    whatever happens to it, the bench line is printed."""
    tmpdir = tempfile.mkdtemp(prefix="mirge_gzu_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    unit = os.path.join(tmpdir, "unit.fastq")
    try:
        fastq.tofile(unit)
        code = ("import sys, json, numpy as np; sys.path.insert(0, %r); import bench; "
                "print('INGEST_GZ ' + json.dumps(bench.run_ingest_gz(np.fromfile(sys.argv[1], dtype=np.uint8), int(sys.argv[2]))))" % ROOT)
        try:
            p = subprocess.run([sys.executable, "-B", "-c", code, unit, str(int(threads))], capture_output=True, text=True, timeout=timeout_s)
        except subprocess.TimeoutExpired:
            return {"error": "timed out after %d s" % timeout_s}
        for ln in p.stdout.splitlines():
            if ln.startswith("INGEST_GZ "):
                return json.loads(ln[len("INGEST_GZ "):])
        return {"error": "exit code %d: %s" % (p.returncode, p.stderr.strip()[-300:])}
    finally:
        shutil.rmtree(tmpdir, ignore_errors=True)


def run_dropin(args, dev, lset, libs, fq_dev, cfg_id):
    """The drop-in boundary itself: baking(args, [file], [name], workDir) then bwtAlign(args, df, workDir, ref_db) -- the two
    calls miRge3.0's main() makes -- on one sample of the workload written to /dev/shm (FASTQ file in, pandas DataFrame
    out, run.log written).  Wall clock; reported beside e2e, which feeds the same kernels from a pinned buffer."""
    import shutil
    import tempfile

    from mirge_b200 import digest as DG
    from mirge_b200 import manifoldAlign as MA
    from tests.util import make_args

    tmp = tempfile.mkdtemp(prefix="mirge_dropin_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    try:
        path = os.path.join(tmp, "sample.fastq")
        with open(path, "wb") as fh:
            step = 1 << 30
            for lo in range(0, int(fq_dev.numel()), step):
                fh.write(fq_dev[lo : lo + step].cpu().numpy().tobytes())
        kw = dict(quiet=True, spikeIn=bool(args.spike), threads=host_threads())
        if cfg_id == 2:
            kw.update(nextseq_trim=20, quality_cutoff="20")
        if cfg_id == 3:
            from mirge_b200 import synth

            kw.update(adapters=[("back", synth.QIA_INNER)], uniq_mol_ids="0,12", qiagenumi=True, umiDedup=True)
        a = make_args(**kw)
        out = {}
        for rep in range(2):  # the second pass is the timed one (first: allocator warm-up, page cache)
            t0 = time.perf_counter()
            df, src, trc, tru = DG.baking(a, [path], ["sample"], tmp, device=dev, count_mode=args.count_mode)
            t1 = time.perf_counter()
            df = MA.bwtAlign(a, df, tmp, "miRBase", libraries=lset, device=dev)
            t2 = time.perf_counter()
            out = {"value": round(args.reads / (t2 - t0) / 1e6, 3), "unit": UNIT, "baking_s": round(t1 - t0, 2),
                   "bwtAlign_s": round(t2 - t1, 2), "rows": int(len(df)), "annotated_rows": int((df["annotFlag"] == 1).sum()),
                   "reads": int(src["sample"]), "input": "FASTQ file on /dev/shm", "output": "pandas DataFrame (reference contract)"}
            try:  # the reference's own stage lines (run.log is appended to: the last pass's are the last ones)
                lines = [ln.strip() for ln in open(os.path.join(tmp, "run.log")) if "second(s)" in ln]
                out["run_log"] = lines[-5:]
            except OSError:
                pass
            del df
        return out
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


DUMP_KEYS = 1 << 16  # unique sequences in the sample that --dump-outputs writes row by row
DUMP_ROW_BYTES = 48 << 20  # bound of that sample's rows (text, counts, annotation); the whole-table files add 88 bytes per sample


def sample_fastq(libs, cfg_id, gs, n_reads, multi_sample, device):
    """FASTQ bytes of global sample ``gs`` of the workload, on ``device``: seeded, identical from run to run."""
    import dataclasses

    from mirge_b200 import synth

    rc = dataclasses.replace(synth.CONFIGS[cfg_id], sample_seed=gs if multi_sample else 0)
    gen = synth.ReadGenerator(libs, rc, device)
    gen.gen.manual_seed(2000 + cfg_id + 7919 * gs)
    return gen.fastq(n_reads, first_index=gs * n_reads)


def dump_outputs(out_dir, tab, columns, annot, hit, n_reads):
    """--dump-outputs: the result table of a pass -- unique sequences, their per-sample counts, their annotation -- as .npy
    files.  Whole-table totals, plus every column for a fixed, seeded sample of the sequences taken in bytewise order of
    their text (key ids follow the insertion order of concurrent threads and differ from run to run).
      totals            [reads, unique sequences, annotated sequences]
      keys_per_round    [11]     sequences annotated in round 0..9, last: unannotated
      reads_per_round   [S, 11]  counts of those sequences per sample (the numbers of annotation.report.csv)
      sample_sequences  [K, W]   ASCII codes of the sampled sequences, 0-padded (float32)
      sample_counts     [K, S]   their counts per sample
      sample_annotation [K, 4]   their round (255: none), mismatches, library entry and offset of the hit"""
    from mirge_b200.manifoldAlign import decode_hits

    os.makedirs(out_dir, exist_ok=True)
    n = int(tab.n_keys)
    dev = annot.device
    counts = torch.zeros(len(columns), n, dtype=torch.float64, device=dev)
    for s, (ids, cnt) in enumerate(columns):
        counts[s, ids.long()] = cnt.double()
    rnd = annot[:n].long().clamp(max=10)  # rounds are 0..9; 0xFF (unannotated) -> 10
    reads_per_round = torch.zeros(len(columns), 11, dtype=torch.float64, device=dev).index_add_(1, rnd, counts)
    perm, offsets, data = tab.export_sorted_device()
    lens_all = offsets[1:] - offsets[:-1]
    width = max(int(lens_all.max().item()), 1) if n else 1
    k = min(n, DUMP_KEYS, DUMP_ROW_BYTES // (4 * width + 8 * len(columns) + 8 * 4))
    pos = torch.from_numpy(np.sort(np.random.default_rng(20240).choice(n, k, replace=False))).to(dev)
    sel, lo, lens = perm[pos], offsets[pos], lens_all[pos]
    col = torch.arange(width, device=dev)
    text = torch.where(col < lens[:, None], data[(lo[:, None] + col).clamp(max=data.numel() - 1)], 0)
    rounds, mm, ref, off = decode_hits(annot[sel].cpu().numpy(), hit[sel].cpu().numpy())
    out = {
        "totals": np.array([n_reads, n, int((rnd < 10).sum().item())], dtype=np.float64),
        "keys_per_round": torch.bincount(rnd, minlength=11).double().cpu().numpy(),
        "reads_per_round": reads_per_round.cpu().numpy(),
        "sample_sequences": text.float().cpu().numpy(),
        "sample_counts": counts[:, sel].T.contiguous().cpu().numpy(),
        "sample_annotation": np.stack([rounds, mm, ref, off], axis=1).astype(np.float64),
    }
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_b200(args):
    import torch.distributed as dist

    import mirge_b200  # noqa: F401
    from mirge_b200 import device as D
    from mirge_b200 import digest as DG
    from mirge_b200 import distributed as MD
    from mirge_b200 import libraries as LB
    from mirge_b200 import manifoldAlign as MA
    from mirge_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        if args.dump_outputs:
            raise SystemExit("bench: --dump-outputs writes the table of one process; run it with one GPU")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = D.Device(local)
    torch.cuda.set_device(dev.tdev)
    batch_bytes = args.batch_mb << 20

    t_setup = time.perf_counter()
    cfg_id = args.config
    libs = synth.make_libraries(mrna_count=args.mrna)
    lset = LB.LibrarySet.from_fasta_dict(dev, libs.fasta_dict())
    cfg = synth.trim_config_for(cfg_id, args.count_mode)
    eng = D.DigestEngine(dev, cfg)
    umi = cfg.umi()
    # this GPU's samples (C4: per-sample abundance perturbation, synth.ReadConfig.sample_seed); resident in HBM
    fqs = [sample_fastq(libs, cfg_id, rank * args.samples + s_i, args.reads, args.samples > 1, dev.tdev) for s_i in range(args.samples)]
    rc = synth.CONFIGS[cfg_id]
    torch.cuda.synchronize()
    nbytes = int(sum(f.numel() for f in fqs))
    reads_per_gpu = args.reads * args.samples
    setup_s = time.perf_counter() - t_setup

    table = D.CollapseTable(dev, min_keys=1 << 22)
    first_level = D.CollapseTable(dev, min_keys=1 << 22) if umi is not None else None
    # N > 1: one exchange per sample after its local collapse.  (--overlap-exchange, single-sample configs: the exchange of
    # every batch on a worker thread / side stream while the next batch is trimmed into a second local table,
    # distributed.ExchangeWorker -- measured slower at N = 2 (61.6 vs 52 ms per pass): five drains / resets of GB-sized
    # tables and two streams of latency-bound kernels that take each other's SM slots cost more than the 12 ms they hide.)
    overlap = world > 1 and args.overlap_exchange and args.samples == 1 and umi is None
    # N > 1, one sample whose reads are spread over the ranks (C2, C5): sharding before the collapse -- every batch's keys go
    # to their owner ranks and are inserted once, there (distributed.ShardedCollapse); --exchange-unique keeps the
    # local-collapse + exchange-of-unique-sequences path that multi-sample and UMI flows use
    sharded = world > 1 and args.samples == 1 and umi is None and not overlap and not args.exchange_unique
    sc = MD.ShardedCollapse(eng, world) if sharded else None
    table_b = D.CollapseTable(dev, min_keys=1 << 22) if overlap else None
    worker = MD.ExchangeWorker(local, world, owner_min_keys=1 << 22) if overlap else None
    owner = worker.owner if worker else (D.CollapseTable(dev, min_keys=1 << 22) if (world > 1 and not sharded) else None)
    state = {}
    xumi = umi if umi is not None else (0, 0)

    def sample_done(columns):
        """the sample's reads are collapsed into `table` (or the first-level table): UMI level, per-sample column,
        exchange to the owners"""
        if umi is not None:
            with dev.timed("drain"):
                ids1, cnt1 = first_level.drain()
            with dev.timed("umi_collapse"):
                DG.umi_collapse(dev, first_level, ids1, cnt1, table, umi, cfg.minimum_length, True)
            first_level.reset()
        with dev.timed("drain"):
            ids, cnt = table.drain()
        if world > 1:
            MD.exchange_and_merge(dev, table, ids, cnt, owner, world, umi=(0, 0))  # (second-level keys carry no UMI)
            with dev.timed("drain"):
                ids, cnt = owner.drain()
        columns.append((ids, cnt))

    def annotate_final(columns):
        tab = owner if owner is not None else table
        keys = MA.KeySet.from_table(tab)
        annot, hit = MA.annotate_keys(dev, lset, keys, args.spike)
        state.update(columns=columns, annot=annot, hit=hit, tab=tab)
        return tab

    def step_resident():
        # (annotating every batch's new keys on a side stream while the next batch is trimmed was measured: no
        # gain for the resident pass -- the kernels do not share SMs usefully -- so the pass stays sequential)
        if overlap:
            # per-batch exchange behind the next batch's trim; the same number of batches on every rank (equal shards)
            worker.reset_owner()
            n = eng.digest_device_exchange(fqs[0], (table, table_b), worker, batch_bytes, n_batches=state["n_batches"])
            worker.finish()
            with dev.timed("drain"):
                ids, cnt = owner.drain()
            annotate_final([(ids, cnt)])
            return n
        table.reset()
        if sharded:
            n = sc.digest_device(fqs[0], table, batch_bytes)
            with dev.timed("drain"):
                ids, cnt = table.drain()
            annotate_final([(ids, cnt)])
            return n
        if owner is not None:
            with dev.timed("owner_reset"):
                owner.reset()
        n, columns = 0, []
        for fq_s in fqs:
            n += eng.digest_device(fq_s, first_level if umi is not None else table, batch_bytes)
            sample_done(columns)
        annotate_final(columns)
        return n

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if overlap:  # every rank submits the same number of per-batch exchanges
        nb = torch.tensor([D.DigestEngine.max_batches(nbytes, batch_bytes)], device=dev.tdev)
        dist.all_reduce(nb, op=dist.ReduceOp.MAX)
        state["n_batches"] = int(nb.item())

    # ---- device-resident throughput ("value")
    for _ in range(args.warmup):
        step_resident()
    barrier()
    dev.timing = True
    dev.timer_totals()
    for k_ in eng.stats:
        eng.stats[k_] = 0
    launches0 = dev.launches
    clocks = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if os.environ.get("MIRGE_B200_EMPTY_CACHE") == "1":
        # profiling runs only (ncu's kernel replay has to save the device memory in use): drop what warm-up left in the
        # allocator.  Not in a measured run -- the timed steps would pay the cudaMalloc calls again (measured: +7 ms per
        # pass at two ranks, +1.3 ms on one GPU)
        torch.cuda.empty_cache()
    torch.cuda.profiler.start()  # ncu --profile-from-start off: the launch list covers exactly the timed region
    e0.record()
    for _ in range(args.steps):
        n_rec = step_resident()
    e1.record()
    barrier()
    torch.cuda.profiler.stop()
    launches = (dev.launches - launches0) // max(args.steps, 1)
    if args.dump_outputs:  # the last timed step's table (before the trace step and the e2e leg, which reuse it)
        dump_outputs(args.dump_outputs, state["tab"], state["columns"], state["annot"], state["hit"], n_rec)
    trace_to = os.environ.get("MIRGE_B200_TRACE")
    if trace_to and rank == 0:
        # diagnostics, outside the timed region: one more step under torch.profiler, kernels / copies per stream in time order
        from torch.profiler import ProfilerActivity, profile

        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            step_resident()
            torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        evs.sort(key=lambda e: e.time_range.start)
        t0 = evs[0].time_range.start if evs else 0
        with open(trace_to, "w") as fh:
            for e in evs:
                fh.write("%10.3f %9.3f ms  stream %-4s %s\n" % ((e.time_range.start - t0) / 1e3, (e.time_range.end - e.time_range.start) / 1e3,
                                                               getattr(e, "device_resource_id", getattr(e, "device_index", "?")), e.name[:90]))
    elif trace_to and world > 1:
        step_resident()  # (the step is collective)
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / max(args.steps, 1)
    timers = dev.timer_totals()
    dev.timing = False
    stats = dict(eng.stats)
    clk = clocks.stop() if clocks else None
    tms = torch.tensor([ms], device=dev.tdev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_max = float(tms.item())
    assert n_rec == reads_per_gpu, (n_rec, reads_per_gpu)
    n_unique = int(state["tab"].n_keys)
    n_annot = int((state["annot"] != 0xFF).sum().item())

    # ---- end to end from pinned host memory
    e2e = None
    hosts = None
    if not args.no_e2e:
        # the host copy of the input (pinned).  If any rank cannot pin that much memory all ranks skip the e2e leg
        # together (it contains collectives) and the line reports e2e = null.
        try:
            bind_to_gpu_numa_node(local)  # pinned pages and the copy threads on the GPU's own NUMA node where allowed
            hosts = []
            for f in fqs:
                h = torch.empty(int(f.numel()), dtype=torch.uint8).pin_memory()
                h.copy_(f)
                hosts.append(h)
        except (RuntimeError, MemoryError) as exc:
            sys.stderr.write("bench: e2e leg skipped on rank %d: %s\n" % (rank, exc))
            hosts = None
        okf = torch.tensor([0 if hosts is None else 1], device=dev.tdev)
        if world > 1:
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
        if int(okf.item()) == 0:
            hosts = None
    if hosts is not None:
        torch.cuda.synchronize()
        streamer = DG.HostStreamer(eng, args.e2e_batch_mb << 20)

        pinned = {}

        def to_host(name, t):
            """device -> pinned host buffer (kept across steps), asynchronous"""
            n_el = int(t.numel())
            buf = pinned.get(name)
            if buf is None or buf.numel() < n_el or buf.dtype != t.dtype:
                buf = torch.empty(max(int(n_el * 1.25), 1), dtype=t.dtype).pin_memory()
                pinned[name] = buf
            buf[:n_el].copy_(t, non_blocking=True)
            return n_el * t.element_size()

        # single GPU, no UMI level: annotation and the D2H of the result table are streamed piece by piece behind the H2D
        # of the following pieces (the keys of a piece are final as soon as it is collapsed)
        sa = MA.StreamedAnnotator(dev, lset, args.spike) if ((world == 1 or sharded) and umi is None) else None

        def step_e2e():
            table.reset()
            if owner is not None:
                owner.reset()
            n, columns, d2h = 0, [], 0
            if sa is not None:
                sa.reset()
            for h in hosts:
                if sa is not None:
                    n += streamer.run(h, table, on_piece=sa, sharded=sc)
                    with dev.timed("drain"):
                        ids, cnt = table.drain()
                    columns.append((ids, cnt))
                else:
                    n += streamer.run(h, first_level if umi is not None else table)
                    sample_done(columns)
            if sa is not None:
                sa.finish(table)
                d2h += sa.d2h_bytes
                for j, (ids, cnt) in enumerate(columns):
                    d2h += to_host("ids%d" % j, ids) + to_host("cnt%d" % j, cnt)
                torch.cuda.current_stream().synchronize()
                return n, d2h
            tab = annotate_final(columns)
            # result table -> host: packed unique sequences, per-sample (key id, count) columns and annotation
            nk = tab.n_keys
            d2h = to_host("arena", tab.arena[: tab.arena_used]) + to_host("key_ref", tab.key_ref[:nk]) + \
                to_host("annot", state["annot"]) + to_host("hit", state["hit"])
            for j, (ids, cnt) in enumerate(columns):
                d2h += to_host("ids%d" % j, ids) + to_host("cnt%d" % j, cnt)
            torch.cuda.current_stream().synchronize()
            return n, d2h

        for _ in range(min(args.warmup, 2)):
            step_e2e()
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(args.steps):
            _, d2h = step_e2e()
        f1.record()
        barrier()
        ems = f0.elapsed_time(f1) / max(args.steps, 1)
        tme = torch.tensor([ems], device=dev.tdev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tme, op=dist.ReduceOp.MAX)
        e2e = {"value": round(reads_per_gpu * world / (float(tme.item()) / 1e3) / 1e6, 3), "unit": UNIT,
               "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": int(d2h), "ms_per_step": round(float(tme.item()), 3)}
        # what the box gives all N ranks at once: the same pinned input copied to the device with no kernel in the way
        # (all ranks start together, max over ranks) -- e2e is bounded by max(this, the device-resident pass)
        try:
            probe = torch.empty(min(int(hosts[0].numel()), 2 << 30), dtype=torch.uint8, device=dev.tdev)
            reps = max(1, min(4, int(nbytes // max(probe.numel(), 1))))
            for timed_pass in (False, True):
                barrier()
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                for _ in range(reps):
                    probe.copy_(hosts[0][: probe.numel()], non_blocking=True)
                g1.record()
                barrier()
            tp = torch.tensor([g0.elapsed_time(g1)], device=dev.tdev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            gbs = reps * probe.numel() / (float(tp.item()) / 1e3) / 1e9
            e2e["h2d_ceiling_gbs_per_gpu"] = round(gbs, 2)
            e2e["h2d_floor_ms_per_step"] = round(nbytes / gbs / 1e6, 3)
            e2e["frac_of_h2d_ceiling"] = round(e2e["h2d_floor_ms_per_step"] / e2e["ms_per_step"], 3)
            del probe
        except RuntimeError as exc:
            sys.stderr.write("bench: H2D ceiling probe skipped: %s\n" % exc)
        del hosts, streamer

    # ---- the reference's own entry points on one sample: baking(args, [file]) + bwtAlign(args, df)  (rank 0, N = 1)
    dropin = None
    if args.dropin and world == 1:
        dropin = run_dropin(args, dev, lset, libs, fqs[0], cfg_id)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (CUDA events on the launch stream, timed region above)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    E = eng.E
    rec_bytes = nbytes / reads_per_gpu
    steps = max(args.steps, 1)
    kinfo = {}
    for name, (cnt_l, tot_ms) in timers.items():
        kinfo[name] = {"launches_per_step": cnt_l // steps, "ms_per_step": round(tot_ms / steps, 3)}
    # algorithmic bytes per read (SURVEY.md section 8d): trim R + 8E ; collapse sum over emitted keys (2K + 16)
    b_trim = rec_bytes + 8 * E
    trim_ms = timers.get("trim", (0, 0.0))[1] / steps
    col_ms = timers.get("collapse", (0, 0.0))[1] / steps
    ann_ms = sum(v[1] for k, v in timers.items() if k.startswith("annotate")) / steps
    kinfo["annotate"] = {"launches_per_step": sum(v[0] for k, v in timers.items() if k.startswith("annotate")) // steps,
                         "ms_per_step": round(ann_ms, 3)}
    trim_gbs = reads_per_gpu * b_trim / (trim_ms / 1e3) / 1e9 if trim_ms else 0.0
    kinfo.setdefault("trim", {})["achieved_gbs"] = round(trim_gbs, 1)
    kinfo["trim"]["frac_hbm"] = round(trim_gbs / peak, 4)
    # collapse: every emitted key is read once and probes/updates one slot: sum over keys of (2K + 16) bytes
    b_col_total = (2 * 4 * stats["key_words"] + 16 * stats["emitted"]) / steps
    col_gbs = b_col_total / (col_ms / 1e3) / 1e9 if col_ms else 0.0
    kinfo.setdefault("collapse", {})["achieved_gbs"] = round(col_gbs, 1)
    kinfo["collapse"]["frac_hbm"] = round(col_gbs / peak, 4)
    kinfo["collapse"]["algorithmic_bytes_per_read"] = round(b_col_total / reads_per_gpu, 1)
    kinfo["trim"]["dp_search_frac"] = round(stats.get("dp_reads", 0) / max(stats["records"], 1), 4)
    kinfo["trim"]["cost_column_frac"] = round(stats.get("dp_redo", 0) / max(stats["records"], 1), 4)
    kinfo["trim"]["second_pass_frac"] = round(stats.get("deferred", 0) / max(stats["records"], 1), 4)
    dom = max((("trim", trim_ms), ("collapse", col_ms), ("annotate", ann_ms)), key=lambda kv: kv[1])[0]
    traffic = None
    traffic_file = "r2_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r2_traffic.json")) else "r1_traffic.json"
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", traffic_file)))["trim_kernel"]
        traffic = int(tr["bytes_per_read"] * reads_per_gpu / max(kinfo["trim"].get("launches_per_step", 1), 1))
    except Exception:
        pass
    roofline = {"kernel": "trim_kernel", "bound": "hbm", "achieved": round(trim_gbs, 1), "peak": peak, "unit": "GB/s",
                "frac": round(trim_gbs / peak, 4), "traffic": traffic,
                "traffic_source": "ncu dram bytes per read (profiles/%s) x reads per launch" % traffic_file,
                "peak_source": peak_src,
                "algorithmic_bytes_per_read": round(b_trim, 1), "dominant_by_time": dom,
                "launches_per_step": kinfo["trim"].get("launches_per_step")}

    # ---- CPU baseline on a bounded sample of the same bytes (rank 0, N = 1 only)
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        sample = min(args.cpu_sample or 12_000_000, args.reads)
        sb = int(sample * rec_bytes * 1.02) + 4096
        raw = fqs[0][: min(sb, int(fqs[0].numel()))].cpu().numpy()
        # cut at the end of read `sample`
        nl = np.flatnonzero(raw == 10)
        raw = raw[: int(nl[4 * sample - 1]) + 1] if nl.size >= 4 * sample else raw[: int(nl[(nl.size // 4) * 4 - 1]) + 1]
        sample = min(sample, nl.size // 4)
        cpu = CpuPath(libs, cfg, threads)
        cpu.step(raw[: int(nl[4 * max(sample // 8, 1) - 1]) + 1], args.spike)  # warm-up on a record-aligned prefix
        t0 = time.perf_counter()
        cpu.step(raw, args.spike)
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": round(sample / dt / 1e6, 4), "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": "first %d reads of the same synthetic workload, oracle port of cutadapt+bowtie semantics, %d threads, %.1f s"
                                  % (sample, threads, dt)}

    # ---- host ingest of compressed input (rank 0, N = 1 only): the first 48 MB of the workload's FASTQ, repeated, as one
    # gzip stream through the chunk-parallel decoder
    ingest_gz = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            head = fqs[0][: min(48 << 20, int(fqs[0].numel()))].cpu().numpy()
            nl_h = np.flatnonzero(head == 10)
            head = head[: int(nl_h[(nl_h.size // 4) * 4 - 1]) + 1]
            ingest_gz = run_ingest_gz_guarded(head, host_threads())
        except Exception as exc:  # a host-side extra must never cost the bench line
            ingest_gz = {"error": "%s: %s" % (type(exc).__name__, exc)}

    value = reads_per_gpu * world / (ms_max / 1e3) / 1e6
    line = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(ms_max, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int32",
        "data": "synthetic",
        "config": {"workload": args.workload, "reads_per_gpu": reads_per_gpu, "samples_per_gpu": args.samples, "read_len": rc.L,
                   "count_mode": args.count_mode,
                   "fastq_bytes_per_gpu": nbytes, "l2": "inputs (%.1f GB per pass) larger than L2" % (nbytes / 1e9),
                   "batch_mb": args.batch_mb, "unique_sequences": n_unique, "annotated_sequences": n_annot,
                   "emission_slots_per_read": E, "setup_s": round(setup_s, 1)},
        "e2e": e2e, "dropin": dropin, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
        "ingest_gz": ingest_gz, "kernels": kinfo,
        "clocks": clk, "bit_exact": "tests/ -m gpu (oracle parity); bench does not re-check",
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse_args()
    # the contract is ONE JSON line on stdout: libraries that print there (NCCL's version banner under
    # NCCL_DEBUG=VERSION, for one) are sent to stderr for the duration of the run
    real_stdout = os.dup(1)
    sys.stdout.flush()
    os.dup2(2, 1)
    import io

    buf = io.StringIO()
    old, sys.stdout = sys.stdout, buf
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_b200(args)
    finally:
        sys.stdout = old
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    out = buf.getvalue()
    if out:
        sys.stdout.write(out)
        sys.stdout.flush()


if __name__ == "__main__":
    main()
