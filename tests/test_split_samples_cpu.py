"""baking_sharded's per-sample driver on CPU / gloo: every sample is digested by all ranks.  distributed.sample_sources
cuts a plain FASTQ file into record-aligned byte ranges (one per rank, possibly empty) and gives a compressed file whole
to rank s % world; the ranks' records go through the ShardedCollapse round protocol (numpy stand-ins for the kernels,
owner = hash of the UMI centre with UMIs), the second UMI level runs on the owner, rank 0 writes the -tcf / -udd rows it
gathers (digest.write_tcf_rows / umi_csv_rows), and the counters are all-reduced -- against a single-process dict
reference."""
import gzip
import multiprocessing as mp
import os
import zlib

import numpy as np
import pytest
import torch
import torch.distributed as dist

from mirge_b200 import digest as DG
from mirge_b200 import distributed as MD
from tests.test_distributed_cpu import SimSharded, _Br, free_port, key_words

CODE = {"A": 0, "C": 1, "G": 2, "T": 3}


def pack(s: str):
    words = [len(s)]
    for w in range((len(s) + 15) // 16):
        v = sum(CODE[c] << (2 * q) for q, c in enumerate(s[16 * w : 16 * w + 16]))
        words.append(v - (1 << 32) if v >= 1 << 31 else v)
    return words


def unpack(words) -> str:
    n = int(words[0]) & 0xFFFF
    return "".join("ACGT"[((int(words[1 + j // 16]) & 0xFFFFFFFF) >> (2 * (j % 16))) & 3] for j in range(n))


def centre(s: str, umi):
    f, b = umi
    return s[f : len(s) - b] if b else s[f:]


class SimCentre(SimSharded):
    """SimSharded with the owner of mirge_shard_scatter_centre: the hash of the key without its UMI flanks."""

    def owner(self, kw):
        s = unpack(kw)
        return zlib.crc32((centre(s, self.umi) if self.umi else s).encode()) % self.world

    def pack(self, br, cap_items=0, cap_words=0):
        W = self.world
        items = [] if br is None else br["items"]
        cap_items = max(int(cap_items), len(items) + 1)
        cap_words = max(int(cap_words), sum(key_words(int(br["keys"][o])) for o, _ in items) + 1 if items else 1)
        out_items = torch.zeros(W * cap_items, dtype=torch.int64)
        out_keys = torch.zeros(W * cap_words, dtype=torch.int32)
        cur_i, cur_w = [0] * W, [0] * W
        for o, c in items:
            kw = br["keys"][o : o + key_words(int(br["keys"][o]))]
            d = self.owner(kw)
            out_items[d * cap_items + cur_i[d]] = cur_w[d] | (c << 32)
            out_keys[d * cap_words + cur_w[d] : d * cap_words + cur_w[d] + len(kw)] = torch.from_numpy(np.asarray(kw, dtype=np.int32))
            cur_i[d] += 1
            cur_w[d] += len(kw)
        cursors = torch.tensor([(i << 32) | w for i, w in zip(cur_i, cur_w)], dtype=torch.int64)
        return {"items": out_items, "keys": out_keys, "cursors": cursors, "cap_items": cap_items, "cap_words": cap_words, "br": br}


def records(data: bytes):
    lines = data.split(b"\n")
    return [lines[i].decode() for i in range(1, len(lines) - 1, 4)]


def batches(src, batch_records=7):
    """The stand-in of HostStreamer + trim: the reads of a source, a few records per batch, key = the read."""
    if src is None:
        return []
    seqs = records(src.read())
    out = []
    for a in range(0, len(seqs), batch_records):
        words, items = [], []
        for s in seqs[a : a + batch_records]:
            items.append((len(words), 1))
            words.extend(pack(s))
        out.append(_Br(keys=np.asarray(words, dtype=np.int64).astype(np.int32), items=items, n_records=len(items)))
    return out


def write_inputs(tmp, rng):
    """plain (many records), plain with one record (empty ranges), gzip; reads of 20-40 bases over a small pool"""
    pool = ["".join(rng.choice(list("ACGT"), int(rng.integers(20, 41)))) for _ in range(30)]
    paths = []
    for name, n, gz in (("a", 400, False), ("one", 1, False), ("c", 150, True), ("d", 97, False)):
        data = "".join("@%s.%d\n%s\n+\n%s\n" % (name, k, s, "I" * len(s)) for k, s in
                       enumerate(pool[int(i)] for i in rng.integers(0, len(pool), n))).encode()
        p = os.path.join(tmp, name + (".fastq.gz" if gz else ".fastq"))
        with (gzip.open(p, "wb") if gz else open(p, "wb")) as fh:
            fh.write(data)
        paths.append(p)
    return paths


def driver(rank, world, port, paths, out_dir, umi, q):
    import types

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        eng = types.SimpleNamespace(dev=types.SimpleNamespace(tdev=torch.device("cpu")), stats={})
        sc = SimCentre(eng, world, umi=umi)
        names = [os.path.basename(p).split(".")[0] for p in paths]
        n_read = np.zeros(len(paths), dtype=np.int64)
        trimmed, unique, owned = np.zeros(len(paths), dtype=np.int64), np.zeros(len(paths), dtype=np.int64), {}
        for s, src in MD.sample_sources(paths, rank, world):
            table = {"arena": torch.zeros(64, dtype=torch.int32), "used": 0, "counts": {}}
            try:
                bs = batches(src)
            finally:
                if src is not None:
                    src.close()
            more_any = True
            for i, b in enumerate(bs):
                more_any = sc.round(table, b, i + 1 < len(bs))
                n_read[s] += b.n_records
            sc.drain_rounds(table, more_any)
            first = {unpack(k): c for k, c in table["counts"].items()}
            for k in first:
                assert SimCentre.owner(sc, pack(k)) == rank
            if umi is not None:
                # the second level on the owner (dedup: one per first-level key)
                keys = np.array([k.encode() for k in first] or [b""], dtype="S64")[: len(first)]
                rows = DG.umi_csv_rows(keys, np.array(list(first.values()), dtype=np.int64), umi, 16)
                got = MD.gather_arrays([np.frombuffer(rows.encode("latin-1"), dtype=np.uint8)], 0)
                if got is not None:
                    DG.write_umi_csv_rows(os.path.join(out_dir, names[s] + "_umiCounts.csv"),
                                          "".join(g[0].tobytes().decode("latin-1") for g in got))
                second = {}
                for k in first:
                    c = centre(k, umi)
                    if len(c) >= 16:
                        second[c] = second.get(c, 0) + 1
                final = second
            else:
                final = first
            owned[names[s]] = final
            trimmed[s], unique[s] = sum(final.values()), len(final)
            karr = np.array([k.encode() for k in final], dtype="S64") if final else np.zeros(0, dtype="S1")
            got = MD.gather_arrays([karr, np.array(list(final.values()), dtype=np.int64)], 0)
            if got is not None:
                width = max(g[0].dtype.itemsize for g in got)
                DG.write_tcf_rows(out_dir, names[s], np.concatenate([g[0].astype("S%d" % width) for g in got]),
                                  np.concatenate([g[1] for g in got]))
        tot = torch.from_numpy(np.stack([n_read, trimmed, unique]))
        dist.all_reduce(tot)
        q.put((rank, tot.numpy().tolist(), owned, sc.rounds))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("umi", [None, (4, 4)])
@pytest.mark.parametrize("world", [2, 3])
def test_split_sample_driver_matches_single_process(tmp_path, world, umi):
    paths = write_inputs(str(tmp_path), np.random.default_rng(5))
    out_dir = str(tmp_path / "out")
    os.makedirs(out_dir)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = free_port()
    procs = [ctx.Process(target=driver, args=(r, world, port, paths, out_dir, umi, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = dict((r[0], r[1:]) for r in (q.get(timeout=120) for _ in range(world)))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    names = [os.path.basename(p).split(".")[0] for p in paths]
    n_read, trimmed, unique = res[0][0]
    assert all(res[r][0] == res[0][0] for r in range(world)) and all(res[r][2] == res[0][2] for r in range(world))
    for s, (name, path) in enumerate(zip(names, paths)):
        data = (gzip.open(path).read() if path.endswith(".gz") else open(path, "rb").read())
        reads = records(data)
        first = {}
        for r_ in reads:
            first[r_] = first.get(r_, 0) + 1
        exp = first
        if umi is not None:
            exp = {}
            for k in first:
                c = centre(k, umi)
                if len(c) >= 16:
                    exp[c] = exp.get(c, 0) + 1
            rows = open(os.path.join(out_dir, name + "_umiCounts.csv")).read().split("\n")
            ref = DG.umi_csv_rows(np.array([k.encode() for k in first], dtype="S64"), np.array(list(first.values())), umi, 16)
            assert rows[0] == "UMISeq,transcriptSeq,UMICounts" and sorted(rows[1:]) == sorted(ref.split("\n"))
        # every sequence on exactly one owner; union = the single-process table
        union = {}
        for r in range(world):
            part = res[r][1][name]
            assert not set(part) & set(union)
            union.update(part)
        assert union == exp, name
        assert (n_read[s], trimmed[s], unique[s]) == (len(reads), sum(exp.values()), len(exp))
        lines = open(os.path.join(out_dir, name + ".trim.collapse.fa")).read().split("\n")
        recs = [(int(h.rsplit("_", 1)[1]), q_) for h, q_ in zip(lines[0::2], lines[1::2]) if h]
        assert [c for c, _ in recs] == sorted((c for c, _ in recs), reverse=True)
        assert sorted(recs) == sorted((c, k) for k, c in exp.items())


@pytest.mark.parametrize("world", [2, 3])
def test_sample_sources_cut_plain_files_and_deal_compressed_ones(tmp_path, world):
    """Plain files: the ranks' byte ranges are record-aligned and together the file (the one-record file leaves ranks
    with nothing); a gzip file: the whole stream on rank s % world, nothing elsewhere."""
    paths = write_inputs(str(tmp_path), np.random.default_rng(9))
    got = [[None] * world for _ in paths]
    for r in range(world):
        for s, src in MD.sample_sources(paths, r, world):
            if src is not None:
                got[s][r] = src.read()
                src.close()
    for s, path in enumerate(paths):
        if path.endswith(".gz"):
            assert [r for r in range(world) if got[s][r] is not None] == [s % world]
            assert got[s][s % world] == gzip.open(path).read()
        else:
            assert all(g is not None for g in got[s])
            assert b"".join(got[s]) == open(path, "rb").read()
            assert all(g == b"" or g.startswith(b"@") for g in got[s])
    assert sum(g == b"" for g in got[1]) == world - 1
