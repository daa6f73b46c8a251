"""Every sample digested by all ranks (distributed.baking_sharded over ShardedCollapse) on the GPU: the scatter by UMI
centre (mirge_shard_scatter_centre), the copying receive of the owner tables, and the entry points under torchrun
against the single-process ones (tests/multi_gpu_split_check.py)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import coracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def dev():
    from mirge_b200 import device as D

    return D.Device(0)


def umi_config(name):
    from mirge_b200 import params as P
    from mirge_b200 import synth

    if name == "umi44":  # -umi 4,4: the 4 first and 4 last bases of the trimmed read are the UMI
        return P.TrimConfig(adapters=[("back", synth.ILLUMINA)], uniq_mol_ids="4,4"), 1
    return synth.trim_config_for(3), 3  # --qiagenumi -umi 0,12


def shard_bytes(fq, cuts):
    """The FASTQ bytes of record ranges [cuts[r], cuts[r + 1]) on the device."""
    nl = np.flatnonzero(fq == 10)
    out = []
    for lo, hi in zip(cuts[:-1], cuts[1:]):
        b0 = 0 if lo == 0 else int(nl[4 * lo - 1]) + 1
        b1 = 0 if hi == 0 else int(nl[4 * hi - 1]) + 1
        out.append(torch.from_numpy(fq[b0:b1].copy()).to("cuda"))
    return out


def loopback_rounds(eng, scs, tables, shards, batch=2 << 20):
    """ShardedCollapse's rounds for len(scs) ranks in one process: every rank's batch is packed, the pieces each owner
    receives are put where the owner's receive puts them (end of its arena, or a buffer of the round once repeats
    dominate: copies_keys), and inserted.  Returns (records, rounds that received in place, rounds that copied)."""
    from mirge_b200 import distributed as MD

    world = len(scs)
    pos = [0] * world
    n_rec = in_place = copied = 0
    while any(pos[r] < shards[r].numel() for r in range(world)):
        packed, sizes = [], []
        for r in range(world):
            br = None
            if pos[r] < shards[r].numel():
                end = min(int(shards[r].numel()), pos[r] + batch)
                final = end == shards[r].numel()
                br = eng.trim_batch(shards[r][pos[r] : end], end - pos[r], final, keep=False, table=None)
                pos[r] += br.consumed if not final else end - pos[r]
                n_rec += br.n_records
            p = scs[r].pack(br)
            p = scs[r].settle(p, p["cursors"].cpu().numpy())
            packed.append(p)
            sizes.append(MD.ShardedCollapse.split_cursors(p["cursors"].cpu().numpy()))
        for o in range(world):
            recv_it = [sizes[s][0][o] for s in range(world)]
            recv_w = [sizes[s][1][o] for s in range(world)]
            copy = scs[o].copies_keys(tables[o])
            if copy:
                items, keys, bases = scs[o].place_copy(recv_it, recv_w)
            else:
                items, keys, bases = scs[o].place(tables[o], recv_it, recv_w)
            ai = aw = 0
            for s in range(world):
                ci, cw = packed[s]["cap_items"], packed[s]["cap_words"]
                items[ai : ai + recv_it[s]].copy_(packed[s]["items"][o * ci : o * ci + recv_it[s]])
                keys[aw : aw + recv_w[s]].copy_(packed[s]["keys"][o * cw : o * cw + recv_w[s]])
                ai += recv_it[s]
                aw += recv_w[s]
            if copy:
                scs[o].insert_copy(tables[o], items, recv_it, bases, keys)
                copied += 1
            else:
                scs[o].insert(tables[o], items, recv_it, bases)
                in_place += 1
    return n_rec, in_place, copied


def drained(table):
    ids, cnt = table.drain()
    keys = table.export_keys()
    return ids, cnt, {keys[i].decode("latin-1"): int(c) for i, c in zip(ids.cpu().tolist(), cnt.cpu().tolist())}


@pytest.mark.parametrize("min_new", [0.0, 2.0])  # never / always the copying receive
@pytest.mark.parametrize("name", ["umi44", "qiagen"])
@pytest.mark.parametrize("world", [2, 3])
def test_centre_scatter_and_copying_receive_match_oracle(dev, world, name, min_new):
    """World ranks on ONE device: the first-level keys of every batch go to the owner of their centre, are received in
    place or copied, and the owners' first-level tables (union) equal the oracle's; each centre has exactly one owner,
    the one mirge_partition_plan gives the key; the owner-local second level (mirge_umi_collapse, with and without
    -udd) equals the oracle's Table.umi_collapse."""
    from mirge_b200 import device as D
    from mirge_b200 import digest as DG
    from mirge_b200 import distributed as MD
    from mirge_b200 import synth

    n_reads = 40_000
    cfg, cfg_id = umi_config(name)
    umi = cfg.umi()
    eng = D.DigestEngine(dev, cfg)
    eng.INPLACE_MIN_NEW = min_new
    fq = synth.ReadGenerator(synth.make_libraries(scale=0.05, mrna_count=100), synth.CONFIGS[cfg_id], "cpu").fastq(n_reads).numpy()
    cuts = [0] + [int(n_reads * f) for f in ((0.6,) if world == 2 else (0.5, 0.85))] + [n_reads]
    scs = [MD.ShardedCollapse(eng, world, overlap=False, umi=umi) for _ in range(world)]
    firsts = [D.CollapseTable(dev, min_keys=1 << 12) for _ in range(world)]
    n_rec, in_place, copied = loopback_rounds(eng, scs, firsts, shard_bytes(fq, cuts))
    assert n_rec == n_reads
    assert (copied == 0) if min_new == 0.0 else (in_place == 0 and copied > 0)
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
    union, centre_owner, pairs = {}, {}, []
    f, b = umi
    for o, t in enumerate(firsts):
        ids, cnt, d = drained(t)
        pairs.append((ids, cnt))
        assert not (set(d) & set(union)), "a first-level key is owned by two ranks"
        union.update(d)
        for k in d:
            c = k[f : len(k) - b] if b else k[f:]
            assert centre_owner.setdefault(c, o) == o, "a centre is split across owners"
        # the owner mirge_partition_plan computes for the same keys
        n = int(ids.numel())
        dest, words = dev.empty(n, torch.int32), dev.empty(n, torch.int32)
        dev.check(dev.lib.mirge_partition_plan(dev.ctx, C.byref(t.struct), D._ptr(ids), n, f, b, world, D._ptr(dest), D._ptr(words),
                                               dev.stream()))
        assert n == 0 or set(dest[:n].cpu().tolist()) == {o}
    assert union == tab.to_dict()
    assert len(set(centre_owner.values())) == world
    for dedup in (False, True):
        second = {}
        for o, t in enumerate(firsts):
            sec = D.CollapseTable(dev, min_keys=1 << 12)
            DG.umi_collapse(dev, t, pairs[o][0], pairs[o][1], sec, umi, cfg.minimum_length, dedup)
            d = drained(sec)[2]
            assert not (set(d) & set(second))
            second.update(d)
        assert second == tab.umi_collapse(f, b, cfg.minimum_length, dedup).to_dict(), dedup


@pytest.mark.parametrize("min_new,max_growth", [(None, 1.5), (0.0, None)])
def test_owner_arena_stays_with_unique_sequences(dev, min_new, max_growth):
    """Five samples of the same reads through the rounds (world 2, one device), owners drained after every sample: with
    the copying receive the owners' arenas after the fifth sample stay within 1.5x of their size after the first; with
    the in-place receive only (min_new 0) every received key rests in the arena and they grow about five-fold."""
    from mirge_b200 import device as D
    from mirge_b200 import distributed as MD
    from mirge_b200 import synth

    n_reads, world = 40_000, 2
    eng = D.DigestEngine(dev, synth.trim_config_for(1))
    if min_new is not None:
        eng.INPLACE_MIN_NEW = min_new
    fq = synth.ReadGenerator(synth.make_libraries(scale=0.05, mrna_count=100), synth.CONFIGS[1], "cpu").fastq(n_reads).numpy()
    shards = shard_bytes(fq, [0, n_reads // 2, n_reads])
    scs = [MD.ShardedCollapse(eng, world, overlap=False) for _ in range(world)]
    owners = [D.CollapseTable(dev, min_keys=1 << 12) for _ in range(world)]
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
    exp = tab.to_dict()
    used = []
    for _ in range(5):
        assert loopback_rounds(eng, scs, owners, shards, batch=1 << 20)[0] == n_reads
        union = {}
        for o in owners:
            union.update(drained(o)[2])
        assert union == exp
        used.append(sum(o.arena_used for o in owners))
    if max_growth is not None:
        assert used[-1] <= max_growth * used[0], used
    else:
        assert used[-1] >= 4 * used[0], used


def run_split_check(world, case):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29640 + 3 * world + ["plain", "umi", "qiagen"].index(case)),
           os.path.join(ROOT, "tests", "multi_gpu_split_check.py"), case]
    p = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert "ok=True" in p.stdout


@pytest.mark.parametrize("case", ["plain", "umi", "qiagen"])
def test_entry_points_one_rank_match_single_process(case):
    """baking_sharded + bwtAlign_sharded under torchrun with one rank (which collapses straight into its own tables,
    without ShardedCollapse): DataFrame, counters, SAM files, -tcf and _umiCounts.csv rows equal to the single-process
    baking + bwtAlign."""
    run_split_check(1, case)


@pytest.mark.parametrize("case", ["plain", "umi", "qiagen"])
def test_entry_points_two_ranks_match_single_process(case):
    """The same with two ranks on two GPUs: plain samples cut into byte ranges (one with fewer records than ranks), a
    gzip sample read by one rank, keys sharded before the collapse."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    run_split_check(2, case)
