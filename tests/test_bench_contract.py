"""bench.py's output contract on the CPU arm (the only arm that runs without a GPU): exactly one JSON line on
stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "20000", "--mrna", "300"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "M reads/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_pass(tmp_path):
    """--dump-outputs: float .npy files of the last timed step's result table, under 64 MB, identical from run to run, agreeing
    with the bench line, and with the C oracle on the same seeded reads (counts, round and hit of every sampled sequence).
    --steps 1 and --steps 3 give the same launches per step: the number of timed steps is the one asked for."""
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from mirge_b200 import libraries as LB
    from mirge_b200 import manifoldAlign as MA
    from mirge_b200 import params as P
    from mirge_b200 import synth
    from oracle import coracle

    reads, mrna = 200000, 300
    dumps, lines = [], []
    for steps in (1, 3):
        out = tmp_path / ("steps%d" % steps)
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--config", "1",
                            "--reads", str(reads), "--mrna", str(mrna), "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert p.returncode == 0, p.stderr[-2000:]
        lines.append(json.loads(p.stdout.strip()))
        assert all(f.suffix == ".npy" for f in out.iterdir())
        dumps.append({f.stem: np.load(f) for f in sorted(out.iterdir())})
        assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    a, b = dumps
    assert sorted(a) == ["keys_per_round", "reads_per_round", "sample_annotation", "sample_counts", "sample_sequences", "totals"]
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert np.array_equal(a[name], b[name]), name
    assert [d["steps"] for d in lines] == [1, 3]
    assert lines[0]["gpu_launches"] == lines[1]["gpu_launches"] > 0
    assert lines[0]["kernels"]["trim"]["launches_per_step"] == lines[1]["kernels"]["trim"]["launches_per_step"] > 0
    d = lines[0]
    assert a["totals"].tolist() == [reads, d["config"]["unique_sequences"], d["config"]["annotated_sequences"]]
    assert a["keys_per_round"].sum() == a["totals"][1] and a["keys_per_round"][:10].sum() == a["totals"][2]

    # the oracle on the same reads: collapse table, then the nine rounds for the sampled sequences
    libs = synth.make_libraries(mrna_count=mrna)
    fq = bench.sample_fastq(libs, 1, 0, reads, False, "cuda").cpu().numpy()
    n, tab = coracle.digest_collapse(fq, P.build_trim_params(synth.trim_config_for(1, "head")))
    exp = tab.to_dict()
    assert n == reads and len(exp) == a["totals"][1] and sum(exp.values()) == a["reads_per_round"].sum()
    seqs = [bytes(r[r > 0].astype(np.uint8)) for r in a["sample_sequences"]]
    assert seqs == sorted(seqs) and len(set(seqs)) == len(seqs) == min(len(exp), bench.DUMP_KEYS)
    assert a["sample_counts"][:, 0].tolist() == [exp[s.decode()] for s in seqs]
    blob = np.frombuffer(b"".join(seqs), dtype=np.uint8)
    off = np.zeros(len(seqs) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([len(s) for s in seqs])
    a_o = np.full(len(seqs), 0xFF, dtype=np.uint8)
    h_o = np.full(len(seqs), 0xFFFFFFFFFFFFFFFF, dtype=np.uint64)
    lut = np.frombuffer(b"ACGTN", dtype=np.uint8)
    pols = LB.round_policies()
    for rnd in range(9):  # config 1: no spike-in round; the indexed search of the bench's CPU baseline (full-size libraries)
        L = libs.libs[LB.ROUND_LIBS[rnd]]
        coracle.annotate_round_indexed(blob, off, coracle.Index(lut[L.codes], L.off.astype(np.uint32)), pols[rnd], a_o, h_o, 8)
    assert (a_o != 0xFF).any()
    assert np.array_equal(a["sample_annotation"], np.stack(MA.decode_hits(a_o, h_o), axis=1).astype(np.float64))


def test_ingest_gz_leg_of_the_bench_line():
    """The host-side `ingest_gz` leg: its input really is ONE gzip member holding ONE DEFLATE stream (what makes the
    parallel decoder necessary), and the leg reports both readers on it."""
    import gzip
    import zlib

    import numpy as np

    sys.path.insert(0, ROOT)
    import bench
    from tests.util import random_fastq

    unit = random_fastq(3000, seed=2)
    blob = bench.single_stream_gzip(unit, 4)
    assert gzip.decompress(blob) == unit * 4
    d = zlib.decompressobj(31)
    assert d.decompress(blob) == unit * 4 and d.eof and d.unused_data == b""  # one member, nothing behind it
    res = bench.run_ingest_gz(np.frombuffer(unit, dtype=np.uint8), 2, target_mb=3)
    assert res["value"] > 0 and res["serial_zlib_mb_s"] > 0 and res["threads"] == 2 and res["fastq_mb"] > 2
