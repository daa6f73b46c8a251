"""Device time of each trim kernel on the bench's workload.

The reads of one bench.py sample (default C2: 50 M reads, `-a illumina -nxt 20 -q 20`, HEAD counting; the bench's seeded
libraries and reads) go through DigestEngine.digest_device in the bench's 2 GiB batches.  One untimed pass, then
``--reps`` passes under torch.profiler (CUDA activity only).  Prints one JSON line: per trim kernel its launches and
device milliseconds per pass (stage 1 `trim_kernel<32, true, 1, true>`, stages 2 / 3 `trim_dp_kernel<true|false>`, the
leftover pass `trim_kernel<32, true, 2, false>`), their sum, and the card's name and power limit read in the same process.

    python profiles/trim_stage_time.py [--tree DIR] [--config C] [--reads N] [--reps R]

``--tree`` imports the package from another checkout (e.g. the parent commit, built with its own
__graft_entry__.build()), so two versions can be compared in one job, alternating."""
import argparse
import json
import os
import subprocess
import sys

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
    ap.add_argument("--config", type=int, default=2, choices=(1, 2, 4, 5))
    ap.add_argument("--reads", type=int, default=0, help="reads (default: the config's)")
    ap.add_argument("--reps", type=int, default=3, help="profiled passes (after one untimed pass)")
    ap.add_argument("--batch-mb", type=int, default=2048)
    a = ap.parse_args()
    tree = os.path.abspath(a.tree)
    sys.path.insert(0, tree)
    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench  # the bench's workload table and sample generator (bench.py of the timed checkout)
    import mirge_b200  # noqa: F401
    from mirge_b200 import device as D
    from mirge_b200 import synth

    c = bench.CONFIG_TABLE[a.config]
    reads = a.reads or c["reads"]
    dev = D.Device(0)
    torch.cuda.set_device(dev.tdev)
    libs = synth.make_libraries(mrna_count=c["mrna"])
    eng = D.DigestEngine(dev, synth.trim_config_for(a.config, "head"))
    fq = bench.sample_fastq(libs, a.config, 0, reads, False, dev.tdev)
    table = D.CollapseTable(dev, min_keys=1 << 22)
    batch = a.batch_mb << 20

    def one_pass():
        table.reset()
        n = eng.digest_device(fq, table, batch)
        torch.cuda.synchronize()
        return n

    n_records = one_pass()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.reps):
            one_pass()
    kernels = {}
    for ev in prof.key_averages():
        name = ev.key.split("(")[0].replace("void ", "").strip()
        if not name.startswith(("trim_kernel", "trim_dp_kernel")):
            continue
        us = getattr(ev, "device_time_total", None)
        if us is None:
            us = ev.cuda_time_total
        k = kernels.setdefault(name, [0, 0.0])
        k[0] += ev.count
        k[1] += us / 1e3
    out = {k: {"launches_per_pass": v[0] // a.reps, "ms_per_pass": round(v[1] / a.reps, 3)} for k, v in sorted(kernels.items())}
    name, power = card()
    print(json.dumps({"tree": tree, "workload": c["label"], "reads": reads, "records": int(n_records), "reps": a.reps,
                      "gpu": name, "power_limit": power, "kernels": out,
                      "trim_ms_per_pass": round(sum(v["ms_per_pass"] for v in out.values()), 3)}))


if __name__ == "__main__":
    main()
