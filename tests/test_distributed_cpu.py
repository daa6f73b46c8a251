"""Host-side logic of the multi-GPU path on CPU (gloo, world_size 2): sharding + the variable-size
record all-to-all (mirge_b200.distributed.exchange_records).  Records are built by the oracle's
collapse here; on GPUs the same plumbing moves records packed by mirge_partition_scatter."""
import os
import socket
import zlib

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import mirge_b200  # noqa: F401
from mirge_b200 import distributed as MD
from mirge_b200 import params as P
from oracle import coracle
from tests.util import CONFIGS, random_fastq


def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def owner_of(key: str, world: int) -> int:
    return zlib.crc32(key.encode()) % world


def pack(records):
    """[(key, count)] -> (int32 words, int32 sizes): record = [count][len][ascii bytes, 4 per word]"""
    words, sizes = [], []
    for k, c in records:
        b = k.encode() + b"\0" * (-len(k) % 4)
        w = [c, len(k)] + list(np.frombuffer(b, dtype=np.int32))
        words.extend(int(x) for x in w)
        sizes.append(len(w))
    return torch.tensor(words, dtype=torch.int32), torch.tensor(sizes, dtype=torch.int32)


def unpack(words, sizes):
    out, o = [], 0
    w = words.numpy()
    for s in sizes.tolist():
        c, ln = int(w[o]), int(w[o + 1])
        out.append((w[o + 2 : o + s].tobytes()[:ln].decode(), c))
        o += s
    return out


def worker(rank, world, port, data, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        cfg = CONFIGS["release"]
        cp = P.build_trim_params(cfg)
        # shard whole records across ranks
        recs = data.split(b"\n@")
        recs = [recs[0]] + [b"@" + r for r in recs[1:]]
        lo, hi = MD.shard_ranges(len(recs), world)[rank]
        shard = b"\n".join(recs[lo:hi])
        if not shard.endswith(b"\n"):
            shard += b"\n"
        _, tab = coracle.digest_collapse(np.frombuffer(shard, dtype=np.uint8), cp)
        local = tab.to_dict()
        by_dest = sorted(local.items(), key=lambda kv: (owner_of(kv[0], world), kv[0]))
        words, sizes = pack(by_dest)
        send = torch.zeros(world, dtype=torch.int64)
        for k, _ in by_dest:
            send[owner_of(k, world)] += 1
        r_words, r_sizes = MD.exchange_records(words, sizes, send)
        merged = {}
        for k, c in unpack(r_words, r_sizes):
            assert owner_of(k, world) == rank
            merged[k] = merged.get(k, 0) + c
        q.put((rank, merged))
    finally:
        dist.destroy_process_group()


def test_shard_ranges():
    assert MD.shard_ranges(10, 3) == [(0, 4), (4, 7), (7, 10)]
    assert MD.shard_ranges(2, 4) == [(0, 1), (1, 2), (2, 2), (2, 2)]
    assert MD.shard_ranges(0, 2) == [(0, 0), (0, 0)]


def test_hash_partitioned_exchange_world2():
    world = 2
    data = random_fastq(1500, seed=9, pool=80)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=worker, args=(r, world, port, data, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    cp = P.build_trim_params(CONFIGS["release"])
    _, tab = coracle.digest_collapse(np.frombuffer(data, dtype=np.uint8), cp)
    exp = tab.to_dict()
    # every unique sequence is owned by exactly one rank and the merged counts equal the global collapse
    assert set(results[0]).isdisjoint(results[1])
    union = {**results[0], **results[1]}
    assert union == exp
    assert len(results[0]) > 0 and len(results[1]) > 0


def gather_worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        rng = np.random.default_rng(50 + rank)
        n = [700, 0, 1300][rank]  # one rank owns nothing
        width = [30, 1, 75][rank]  # the key columns of the ranks differ in width
        keys = np.array(["".join(rng.choice(list("ACGT"), int(rng.integers(1, width + 1)))) for _ in range(n)], dtype="S%d" % width) \
            if n else np.zeros(0, dtype="S1")
        cols = []
        for j in range(3):  # three samples: (ids, counts) of unequal lengths
            m = int(rng.integers(0, n + 1)) if n else 0
            cols += [rng.integers(0, max(n, 1), m).astype(np.int64), rng.integers(1, 1000, m).astype(np.int64)]
        annot = rng.integers(0, 256, n).astype(np.uint8)
        got = MD.gather_arrays([keys] + cols + [annot], 0)
        assert (got is None) == (rank != 0)
        q.put((rank, [keys] + cols + [annot], got))
    finally:
        dist.destroy_process_group()


def test_gather_arrays_world3():
    """The row gather of baking_sharded / bwtAlign_sharded: raw arrays of unequal length (byte-string columns of unequal
    width, an empty rank) arrive at rank 0 as every rank sent them."""
    world = 3
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=gather_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = {}
    for _ in range(world):
        rank, sent, got = q.get(timeout=120)
        res[rank] = (sent, got)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    got = res[0][1]
    assert len(got) == world
    for r in range(world):
        sent = res[r][0]
        assert len(got[r]) == len(sent)
        for a, b in zip(sent, got[r]):
            assert a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a, b), (r, a.dtype, b.dtype)


# ---------------------------------------------------------------------------------------------------------------
# distributed.ShardedCollapse (sharding before the collapse): the round protocol on CPU / gloo.  The three kernels
# (mirge_shard_scatter, the arena placement + mirge_shard_rebase, mirge_collapse_insert_list) are replaced by numpy
# stand-ins with the same buffer layouts; everything else -- pack-first ordering, all-gathered sizes and "more
# input" flags, the exact-size exchange with the rank's own part bypassing it, undersized regions repeated with
# exact sizes, ranks that run out of batches early, the three-stage pipeline and its drain -- is the product code.
# ---------------------------------------------------------------------------------------------------------------


def key_words(header: int) -> int:
    """words of a packed key from its header word (len | n_exc << 16): csrc/key_format.cuh"""
    ln, exc = header & 0xFFFF, header >> 16
    return 1 + (ln + 15) // 16 + exc


def sim_owner(words, world):
    return zlib.crc32(np.asarray(words, dtype=np.int32).tobytes()) % world


class SimSharded(MD.ShardedCollapse):
    def pack(self, br, cap_items=0, cap_words=0):
        W = self.world
        items = [] if br is None else br["items"]
        n_items = len(items)
        n_words = sum(key_words(int(br["keys"][o])) for o, _ in items) if n_items else 0
        cap_items = max(int(cap_items), int(n_items / W * self.slack) + 2)
        cap_words = max(int(cap_words), int(n_words / W * self.slack) + 4)
        out_items = torch.zeros(W * cap_items, dtype=torch.int64)
        out_keys = torch.zeros(W * cap_words, dtype=torch.int32)
        cur_i, cur_w = [0] * W, [0] * W
        for o, c in items:
            nw = key_words(int(br["keys"][o]))
            kw = br["keys"][o : o + nw]
            d = sim_owner(kw, W)
            if cur_i[d] + 1 <= cap_items and cur_w[d] + nw <= cap_words:  # (a full region keeps counting, as the kernel does)
                out_items[d * cap_items + cur_i[d]] = cur_w[d] | (c << 32)
                out_keys[d * cap_words + cur_w[d] : d * cap_words + cur_w[d] + nw] = torch.from_numpy(np.asarray(kw, dtype=np.int32))
            cur_i[d] += 1
            cur_w[d] += nw
        cursors = torch.tensor([(i << 32) | w for i, w in zip(cur_i, cur_w)], dtype=torch.int64)
        return {"items": out_items, "keys": out_keys, "cursors": cursors, "cap_items": cap_items, "cap_words": cap_words, "br": br}

    def place(self, table, recv_items, recv_words):
        n_it, n_w = int(sum(recv_items)), int(sum(recv_words))
        a0 = table["used"]
        if a0 + n_w > table["arena"].numel():
            grown = torch.zeros(2 * (a0 + n_w) + 16, dtype=torch.int32)
            grown[:a0] = table["arena"][:a0]
            table["arena"] = grown
        bases, at = [], a0
        for w in recv_words:
            bases.append(at)
            at += int(w)
        table["used"] = at
        return torch.empty(n_it, dtype=torch.int64), table["arena"][a0:at], bases

    def insert(self, table, items, recv_items, bases, local_br=None):
        arena = table["arena"].numpy()
        lo = 0
        for n, base in zip(recv_items, bases):
            for v in items[lo : lo + n].tolist():
                off, cnt = (v & 0xFFFFFFFF) + base, v >> 32
                kw = tuple(int(x) for x in arena[off : off + key_words(int(arena[off]))])
                table["counts"][kw] = table["counts"].get(kw, 0) + cnt
            lo += n
        table["inserts"] = table.get("inserts", 0) + 1


def sim_batches(rank, n_batches, seed):
    """[{keys: int32 words, items: [(offset, count)]}] of a rank + the (key words -> count) it contributes"""
    rng = np.random.default_rng(seed + 17 * rank)
    pool = [tuple([int(ln)] + [int(x) for x in rng.integers(-2**31, 2**31 - 1, (ln + 15) // 16)]) for ln in rng.integers(16, 60, 40)]
    out, total = [], {}
    for _ in range(n_batches):
        words, items = [], []
        for _ in range(int(rng.integers(1, 60))):
            k = pool[int(rng.integers(len(pool)))] if rng.random() < 0.7 else \
                tuple([33] + [int(x) for x in np.random.default_rng(int(rng.integers(1 << 30))).integers(0, 1 << 20, 3)])
            c = int(rng.integers(1, 4))
            items.append((len(words), c))
            words.extend(k)
            total[k] = total.get(k, 0) + c
        out.append({"keys": np.asarray(words, dtype=np.int64).astype(np.int32), "items": items, "n_records": len(items)})
    return out, total


class _Br(dict):
    n_records = property(lambda self: self["n_records"])


def sharded_worker(rank, world, port, overlap, slack, n_batches, q):
    import types

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        eng = types.SimpleNamespace(dev=types.SimpleNamespace(tdev=torch.device("cpu")), stats={})
        sc = SimSharded(eng, world, overlap=overlap, slack=slack)
        table = {"arena": torch.zeros(64, dtype=torch.int32), "used": 0, "counts": {}}
        pieces = []
        for sample in range(2):  # two samples in a row: the object must come back clean from drain_rounds
            batches, _ = sim_batches(rank, n_batches[rank], 100 * sample)
            more_any = True
            for i, b in enumerate(batches):
                more_any = sc.round(table, _Br(b), i + 1 < len(batches), on_piece=lambda t: pieces.append(len(t["counts"])))
            sc.drain_rounds(table, more_any, on_piece=lambda t: pieces.append(len(t["counts"])))
            assert not sc.q
        q.put((rank, table["counts"], sc.rounds, len(pieces)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("overlap,slack,n_batches", [(True, 1.2, (5, 2)), (False, 1.2, (1, 4)), (True, 0.3, (3, 3)), (True, 1.2, (0, 3))])
def test_sharding_before_collapse_round_protocol_world2(overlap, slack, n_batches):
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=sharded_worker, args=(r, world, port, overlap, slack, n_batches, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = {}
    for _ in range(world):
        rank, counts, rounds, n_pieces = q.get(timeout=120)
        results[rank] = (counts, rounds, n_pieces)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    exp = {}
    for rank in range(world):
        for sample in range(2):
            _, tot = sim_batches(rank, n_batches[rank], 100 * sample)
            for k, c in tot.items():
                exp[k] = exp.get(k, 0) + c
    got0, got1 = results[0][0], results[1][0]
    assert set(got0).isdisjoint(got1)
    assert all(sim_owner(k, world) == 0 for k in got0) and all(sim_owner(k, world) == 1 for k in got1)
    assert {**got0, **got1} == exp
    # both ranks ran the same number of rounds: max(batches) per sample (+ the closing round of the pipelined form,
    # which learns one round late that everybody is done), and every round's arrivals were handed to on_piece
    assert results[0][1] == results[1][1]
    per_sample = max(max(n_batches), 1)
    assert results[0][1] == 2 * per_sample
    assert results[0][2] == results[0][1]


def test_assemble_table_equals_the_reference_join():
    """Rank 0's assembly of the owners' slices (distributed.assemble_table) against the reference's matrix build
    (digest.py:237-261: one column per sample, successive outer joins, fillna(0), flag columns): random per-sample
    tables cut by owner over three ranks, one rank owning nothing, a key no sample counted."""
    import pandas as pd

    from mirge_b200 import digest as DG

    rng = np.random.default_rng(12)
    names = ["a", "b", "c"]
    pool = ["".join(rng.choice(list("ACGT"), int(rng.integers(16, 40)))) for _ in range(400)]
    tables = [{k: int(rng.integers(1, 50)) for k in rng.choice(pool, int(rng.integers(50, 300)), replace=False)} for _ in names]
    world = 3
    owner = lambda k: 0 if zlib.crc32(k.encode()) % 2 == 0 else 2  # rank 1 owns nothing
    gathered = []
    for r in range(world):
        keys = sorted({k for t in tables for k in t if owner(k) == r})
        if r == 0:
            keys.append("TTTTTTTTTTTTTTTTTTTT")  # in the owner's table (an earlier sample of the run), counted by none of these
        rng.shuffle(keys)
        kid = {k: i for i, k in enumerate(keys)}
        width = max([len(k) for k in keys] + [1])
        karr = np.array([k.encode() for k in keys], dtype="S%d" % width) if keys else np.zeros(0, dtype="S1")
        ps = []
        for t in tables:
            mine = [(kid[k], c) for k, c in t.items() if owner(k) == r]
            ps.append((np.array([i for i, _ in mine], dtype=np.int64), np.array([c for _, c in mine], dtype=np.int64)))
        gathered.append((karr, ps))
    df, order, offs, n_all = MD.assemble_table(gathered, names)
    # the reference's way
    ref = None
    for n, t in zip(names, tables):
        col = pd.DataFrame(list(t.items()), columns=["Sequence", n]).set_index("Sequence")
        ref = col if ref is None else ref.join(col, how="outer")
    ref = ref.fillna(0).astype(int)
    ref = ref.assign(**dict.fromkeys(DG.INITIAL_FLAGS, "")).assign(annotFlag=0)
    ref = ref.reindex(columns=["annotFlag"] + DG.INITIAL_FLAGS + names).astype({"annotFlag": int})
    assert list(df.index) == list(ref.index) and list(df.columns) == list(ref.columns)
    assert df.to_csv() == ref.to_csv()
    assert [str(t) for t in df.dtypes] == [str(t) for t in ref.dtypes] and df.index.name == "Sequence"
    # the Arrow-backed form large tables take (no Python object per row) writes the same file
    import mirge_b200.digest as DGm

    old_min, DGm.ARROW_INDEX_MIN = DGm.ARROW_INDEX_MIN, 10
    try:
        df2 = MD.assemble_table(gathered, names)[0]
    finally:
        DGm.ARROW_INDEX_MIN = old_min
    assert df2.to_csv() == ref.to_csv() and list(df2.index) == list(ref.index)
    empty = MD.assemble_table([(np.zeros(0, dtype="S1"), [(np.zeros(0, dtype=np.int64),) * 2] * 3)] * 2, names)[0]
    assert len(empty) == 0 and list(empty.columns) == list(ref.columns)
    assert n_all == sum(len(g[0]) for g in gathered) and len(order) == len(ref) and list(offs) == [0, len(gathered[0][0]), len(gathered[0][0]), n_all]


def test_fill_annotation_places_the_owners_results_in_table_order():
    """bwtAlign_sharded's rank-0 half (distributed.fill_annotation): rounds and reference indices arrive in gather order
    (rank by rank, each rank's keys in its own order), the table is in lexicographic order with unseen keys dropped; every
    row must get the name of ITS sequence's hit, annotFlag 1 iff annotated, and the spike-in column only with -spk."""
    rng = np.random.default_rng(31)
    names = ["s1", "s2"]
    world = 3
    gathered, truth = [], {}
    names_of = {rnd: ["lib%d_ref%d" % (rnd, i) for i in range(50)] for rnd in range(10)}
    annot_parts, ref_parts = [], []
    for r in range(world):
        keys = ["".join(rng.choice(list("ACGT"), int(rng.integers(16, 30)))) for _ in range(int(rng.integers(0, 200)))]
        keys = sorted(set(keys), key=lambda k: rng.random())
        karr = np.array([k.encode() for k in keys], dtype="S30") if keys else np.zeros(0, dtype="S1")
        ps = []
        for _ in names:
            ids = np.array(sorted(rng.choice(len(keys), int(rng.integers(0, len(keys) + 1)), replace=False)), dtype=np.int64) if keys else np.zeros(0, dtype=np.int64)
            ps.append((ids, rng.integers(1, 99, ids.size).astype(np.int64)))
        gathered.append((karr, ps))
        annot = rng.choice(np.array([0xFF, 0xFF, 0, 1, 2, 5, 8, 9], dtype=np.uint8), len(keys)).astype(np.uint8)
        ref = rng.integers(0, 50, len(keys)).astype(np.int64)
        ref[annot == 0xFF] = 0xFFFFFFF  # what decode_hits gives for "no hit": must never be used as an index
        annot_parts.append(annot)
        ref_parts.append(ref)
        for k, a, x in zip(keys, annot, ref):
            truth[k] = (int(a), int(x))
    df, order, offs, n_all = MD.assemble_table(gathered, names)
    annot_all, ref_all = np.concatenate(annot_parts), np.concatenate(ref_parts)
    for spike in (True, False):
        ann = annot_all.copy()
        if not spike:
            ann[ann == 9] = 0xFF  # the spike-in round only runs with -spk
        out = MD.fill_annotation(df.copy(), ann, ref_all, order, names_of, spike)
        cols = list(out.columns)
        assert ("spike-in" in cols) == spike and cols[0] == "annotFlag" and cols[-2:] == names
        flag_cols = cols[1:-2]
        assert len(flag_cols) == (10 if spike else 9)
        n_annot = 0
        for seq, row in out.iterrows():
            a, x = truth[seq]
            if a == 9 and not spike:
                a = 0xFF
            assert int(row["annotFlag"]) == (1 if a != 0xFF else 0), seq
            for rnd, c in enumerate(flag_cols):
                assert row[c] == (names_of[rnd][x] if a == rnd else ""), (seq, c)
            n_annot += a != 0xFF
        assert n_annot > 20
