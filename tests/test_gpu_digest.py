"""GPU parity: CUDA tokenise/trim/collapse (through the C ABI) vs the CPU oracle, bit-exact."""
import zlib

import numpy as np
import pytest

from mirge_b200 import abi
from mirge_b200 import params as P
from oracle import coracle
from tests.util import CONFIG_DATA, CONFIGS, ILL, random_fastq

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def dev():
    from mirge_b200 import device as D

    return D.Device(0)


def to_dev(dev, data: bytes, pad_front: int = 0):
    t = torch.frombuffer(bytearray(b"\n" * pad_front + data), dtype=torch.uint8).to(dev.tdev)
    return t[pad_front:]


def table_dict(table):
    ids, cnt = table.drain()
    keys = table.export_keys()
    return {keys[i].decode("latin-1"): int(c) for i, c in zip(ids.cpu().tolist(), cnt.cpu().tolist())}


def gpu_windows(eng, br):
    E = eng.E
    win = br.win.cpu().numpy().view(np.uint16).reshape(br.n_records, E, 4)
    kept = (br.key_off.cpu().numpy().view(np.uint32).reshape(br.n_records, E) != abi.NO_KEY).astype(np.uint8)
    return win, kept


@pytest.mark.parametrize("mode", [0, 1, 2])
@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_trim_and_collapse_match_oracle(dev, name, mode):
    """mode 0: automatic kernel choice (split bit-parallel pipeline where it applies); mode 1: generic full DP;
    mode 2: bit-parallel kernel without the split."""
    from mirge_b200 import device as D

    cfg = CONFIGS[name]
    data = random_fastq(3000, seed=zlib.crc32(name.encode()) % 1000 + 1, n_rate=0.02, lower_rate=0.01,
                        **CONFIG_DATA.get(name, {}))
    fq = np.frombuffer(data, dtype=np.uint8)
    eng = D.DigestEngine(dev, cfg)
    eng.set_trim_mode(mode)
    n, win_o, kept_o = coracle.trim(fq, dev.trim_params)
    buf = to_dev(dev, data)
    br = eng.trim_batch(buf, buf.numel(), True)
    assert br.n_records == n
    win_g, kept_g = gpu_windows(eng, br)
    assert np.array_equal(kept_g, kept_o)
    # windows are defined for every slot (kept or not)
    bad = np.argwhere((win_g != win_o).any(axis=2))
    assert bad.size == 0, "first differing (record, slot): %s gpu=%s oracle=%s" % (
        bad[0], win_g[tuple(bad[0])], win_o[tuple(bad[0])])
    assert br.n_emitted == int(kept_o.sum())
    table = D.CollapseTable(dev, min_keys=256)  # small: exercises growth
    eng.collapse_batch(table, br)
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=2)
    exp = tab.to_dict()
    umi = cfg.umi()
    if umi is None:
        assert table_dict(table) == exp
    else:
        ids, cnt = table.drain()
        for dedup in (False, True):
            second = D.CollapseTable(dev, min_keys=256)
            second.reserve(len(ids), int(table.arena_used))
            deferred = dev.empty(len(ids), torch.int32)
            dev.check(dev.lib.mirge_umi_collapse(dev.ctx, table.struct, ids.data_ptr(), cnt.data_ptr(), len(ids),
                                                 second.struct, umi[0], umi[1], cfg.minimum_length, int(dedup),
                                                 deferred.data_ptr(), dev.stream()))
            t2 = tab.umi_collapse(umi[0], umi[1], cfg.minimum_length, dedup)
            assert table_dict(second) == t2.to_dict()


def test_batching_alignment_and_eof(dev):
    from mirge_b200 import device as D

    cfg = CONFIGS["default"]
    data = random_fastq(5000, seed=77)
    fq = np.frombuffer(data, dtype=np.uint8)
    eng = D.DigestEngine(dev, cfg)
    _, tab = coracle.digest_collapse(fq, dev.trim_params)
    exp = tab.to_dict()
    for pad, batch in ((0, 1 << 30), (0, 20000), (5, 33333), (13, 7777)):
        table = D.CollapseTable(dev, min_keys=1 << 10)
        buf = to_dev(dev, data, pad)
        n = eng.digest_device(buf, table, batch_bytes=batch)
        assert n == 5000
        assert table_dict(table) == exp, (pad, batch)
    # CRLF and missing final newline give the same table
    for variant in (random_fastq(5000, seed=77, crlf=True), data[:-1]):
        table = D.CollapseTable(dev, min_keys=1 << 10)
        buf = to_dev(dev, variant, 3)
        assert eng.digest_device(buf, table, batch_bytes=50000) == 5000
        assert table_dict(table) == exp
    # empty input
    table = D.CollapseTable(dev, min_keys=1 << 10)
    assert eng.digest_device(torch.empty(0, dtype=torch.uint8, device=dev.tdev), table) == 0
    assert table_dict(table) == {}


def test_format_errors(dev):
    from mirge_b200 import device as D

    eng = D.DigestEngine(dev, CONFIGS["default"])
    for bad in (b"@a\nACGT\n+\nIII\n", b"@a\nACGT\n+\n", b"a\nACGT\n+\nIIII\n", b"@a\nACGT\n-\nIIII\n"):
        table = D.CollapseTable(dev, min_keys=1 << 10)
        with pytest.raises(D.FastqFormatError):
            eng.digest_device(to_dev(dev, bad), table)


def test_multi_sample_drain(dev):
    """Two samples through one table: per-sample counts via drain, shared key ids."""
    from mirge_b200 import device as D

    cfg = CONFIGS["release"]
    eng = D.DigestEngine(dev, cfg)
    table = D.CollapseTable(dev, min_keys=1 << 10)
    exp = []
    got = []
    for seed in (1, 2):
        data = random_fastq(2000, seed=seed, pool=50)
        _, tab = coracle.digest_collapse(np.frombuffer(data, dtype=np.uint8), dev.trim_params)
        exp.append(tab.to_dict())
        eng.digest_device(to_dev(dev, data), table)
        got.append(table_dict(table))
    assert got == exp
    assert table.n_keys == len(set(exp[0]) | set(exp[1]))


def test_hot_key_contention(dev):
    """One sequence repeated 200k times + unique ones: exercises the claim/publish/defer path."""
    from mirge_b200 import device as D

    cfg = P.TrimConfig(adapters=[("back", ILL)], count_mode="release")
    eng = D.DigestEngine(dev, cfg)
    rec = b"@r\nTGAGGTAGTAGGTTGTATAGTT" + ILL.encode()[:28] + b"\n+\n" + b"I" * 50 + b"\n"
    data = rec * 200000 + random_fastq(1000, seed=3)
    table = D.CollapseTable(dev, min_keys=1 << 10)
    assert eng.digest_device(to_dev(dev, data), table) == 201000
    got = table_dict(table)
    _, tab = coracle.digest_collapse(np.frombuffer(data, dtype=np.uint8), dev.trim_params, nthreads=4)
    assert got == tab.to_dict()
    assert got["TGAGGTAGTAGGTTGTATAGTT"] >= 200000


@pytest.mark.parametrize("cfg_id", [1, 2, 3, 4, 5])
def test_synthetic_workloads_match_oracle(dev, cfg_id):
    """The benchmark's own read model (SURVEY.md section 8d) at 300k reads: windows and table bit-exact."""
    from mirge_b200 import device as D
    from mirge_b200 import synth

    libs = synth.make_libraries(scale=0.1, mrna_count=200)
    gen = synth.ReadGenerator(libs, synth.CONFIGS[cfg_id], dev.tdev)
    buf = gen.fastq(300_000)
    cfg = synth.trim_config_for(cfg_id)
    eng = D.DigestEngine(dev, cfg)
    fq = buf.cpu().numpy()
    n, win_o, kept_o = coracle.trim(fq, dev.trim_params, nthreads=8)
    br = eng.trim_batch(buf, buf.numel(), True)
    win_g, kept_g = gpu_windows(eng, br)
    assert br.n_records == n == 300_000
    assert np.array_equal(kept_g, kept_o)
    bad = np.argwhere((win_g != win_o).any(axis=2))
    assert bad.size == 0, "first differing (record, slot): %s gpu=%s oracle=%s" % (
        bad[0], win_g[tuple(bad[0])], win_o[tuple(bad[0])])
    table = D.CollapseTable(dev, min_keys=1 << 12)
    eng.collapse_batch(table, br)
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
    assert table_dict(table) == tab.to_dict()


def test_long_records_fall_back_to_generic_kernel(dev):
    """Records too large for the bit-parallel kernel's staging trigger the generic kernel (same results)."""
    from mirge_b200 import device as D

    cfg = CONFIGS["default"]
    eng = D.DigestEngine(dev, cfg)
    rng = np.random.default_rng(4)
    recs = []
    for i in range(300):
        L = int(rng.integers(300, 500))
        s = "".join(rng.choice(list("ACGT"), L))
        if i % 3 == 0:
            s = s[:100] + ILL + s[100 + len(ILL):]
        recs.append("@%s\n%s\n+\n%s\n" % ("h" * 700, s, "I" * L))
    data = "".join(recs).encode()
    table = D.CollapseTable(dev, min_keys=1 << 10)
    assert eng.digest_device(to_dev(dev, data), table) == 300
    _, tab = coracle.digest_collapse(np.frombuffer(data, dtype=np.uint8), dev.trim_params)
    assert table_dict(table) == tab.to_dict()


def test_host_streamer_pipeline_matches_device_path(dev):
    """HostStreamer (pipelined H2D, tails carried in the headroom) vs the resident path, odd piece sizes."""
    import io

    from mirge_b200 import device as D
    from mirge_b200 import digest as DG

    cfg = CONFIGS["default"]
    data = random_fastq(6000, seed=91)
    eng = D.DigestEngine(dev, cfg)
    _, tab = coracle.digest_collapse(np.frombuffer(data, dtype=np.uint8), dev.trim_params)
    exp = tab.to_dict()
    pinned = torch.frombuffer(bytearray(data), dtype=torch.uint8).pin_memory()
    for batch, n_buf, max_record in ((1 << 20, 3, 1 << 12), (50_000, 3, 1 << 12), (7_777, 2, 1 << 10), (301, 4, 1 << 10)):
        for src in (io.BytesIO(data), data, pinned):
            table = D.CollapseTable(dev, min_keys=1 << 10)
            st = DG.HostStreamer(eng, batch, max_record=max_record, n_buf=n_buf)
            seen = []
            n = st.run(src if not isinstance(src, bytes) else DG._BytesSource(src), table, on_piece=lambda t: seen.append(t.n_keys))
            assert n == 6000 and st.h2d_bytes == len(data)
            assert seen == sorted(seen) and seen[-1] == len(exp)
            assert table_dict(table) == exp, (batch, n_buf)
    # a record that does not fit the headroom is a format error, not a silent truncation
    table = D.CollapseTable(dev, min_keys=1 << 10)
    with pytest.raises(D.FastqFormatError):
        long_rec = b"@r\n" + b"A" * 400 + b"\n+\n" + b"I" * 400 + b"\n"
        DG.HostStreamer(eng, 64, max_record=64, n_buf=2).run(io.BytesIO(long_rec * 3), table)


def test_arena_growth_tracks_unique_keys(dev):
    """ADVICE r1: with the trim kernels writing every emitted key into the table's arena, a cohort of samples that
    repeat the same sequences grew the arena with the number of reads.  The engine now switches to a batch key
    buffer + copying insert as soon as repeats dominate a batch, so the arena stops growing."""
    from mirge_b200 import device as D

    cfg = CONFIGS["default"]
    data = random_fastq(4000, seed=5)
    fq = np.frombuffer(data, dtype=np.uint8)
    eng = D.DigestEngine(dev, cfg)
    _, tab = coracle.digest_collapse(fq, dev.trim_params)
    exp = tab.to_dict()
    table = D.CollapseTable(dev, min_keys=1 << 10)
    buf = to_dev(dev, data)
    used = []
    for sample in range(6):
        assert eng.digest_device(buf, table, batch_bytes=200000) == 4000
        table.check()
        used.append(table.arena_used)
        assert table_dict(table) == exp  # drained per sample: every sample counts the same
    assert table.n_keys == len(exp)
    assert used[-1] == used[1], used  # no growth once the repeats are recognised
    assert used[1] <= 2 * used[0]


@pytest.mark.parametrize("case", ["synthetic2", "synthetic1", "batches", "crlf_noeol", "long_headers", "tiny", "truncated"])
def test_digest_edge_inputs_match_oracle(dev, case):
    """DigestEngine against the oracle on awkward inputs: batch sizes just above and below 16 KB multiples with
    misaligned starts, CRLF and a missing final newline at a mid-record batch cut, headers of 1.5-4 KB, 1-3 record
    inputs, a truncated final record (format error)."""
    from mirge_b200 import device as D
    from mirge_b200 import synth

    if case.startswith("synthetic"):
        cfg_id = int(case[-1])
        libs = synth.make_libraries(scale=0.1, mrna_count=200)
        buf = synth.ReadGenerator(libs, synth.CONFIGS[cfg_id], dev.tdev).fastq(200_000)
        eng = D.DigestEngine(dev, synth.trim_config_for(cfg_id))
        fq = buf.cpu().numpy()
        n, win_o, kept_o = coracle.trim(fq, dev.trim_params, nthreads=8)
        br = eng.trim_batch(buf, buf.numel(), True)
        assert br.n_records == n == 200_000
        win_g, kept_g = gpu_windows(eng, br)
        assert np.array_equal(kept_g, kept_o) and np.array_equal(win_g, win_o)
        table = D.CollapseTable(dev, min_keys=1 << 12)
        eng.collapse_batch(table, br)
        _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
        assert table_dict(table) == tab.to_dict()
        return
    eng = D.DigestEngine(dev, CONFIGS["default"])
    if case == "batches":
        data = random_fastq(20000, seed=12, n_rate=0.0005)
        variants = [(data, pad, batch) for pad, batch in ((0, 1 << 30), (0, 16384), (3, 16384 * 3 + 1), (13, 50001), (7, 18432))]
    elif case == "crlf_noeol":
        base = random_fastq(9000, seed=13, n_rate=0.0005)
        variants = [(random_fastq(9000, seed=13, n_rate=0.0005, crlf=True), 5, 1 << 30), (base[:-1], 0, 1 << 30), (base[:-1], 9, 40000)]
        data = base
    elif case == "long_headers":
        rng = np.random.default_rng(8)
        recs = []
        for i in range(400):
            L = int(rng.integers(20, 60))
            s = "".join(rng.choice(list("ACGT"), L))
            hdr = "r%d" % i + ("x" * int(rng.integers(1500, 4000)) if i % 7 == 0 else "")
            seq = (s[:15] + ILL + s)[:L] if i % 2 else s
            recs.append("@%s\n%s\n+\n%s\n" % (hdr, seq, "I" * L))
        data = "".join(recs).encode()
        variants = [(data, 0, 1 << 30), (data, 11, 30000)]
    elif case == "tiny":
        data = b"@a\nTGAGGTAGTAGGTTGTATAGTT\n+\nIIIIIIIIIIIIIIIIIIIIII\n"
        variants = [(data, 0, 1 << 30), (data[:-1], 1, 1 << 30), (data * 3, 2, 1 << 30)]
    else:  # truncated final record: a format error, as with the tokeniser
        data = random_fastq(3000, seed=14, n_rate=0.0005)
        cut = data[: len(data) - 30]
        table = D.CollapseTable(dev, min_keys=1 << 10)
        with pytest.raises(D.FastqFormatError):
            eng.digest_device(to_dev(dev, cut), table)
        return
    for blob, pad, batch in variants:
        ref = data if case != "tiny" else blob + (b"\n" if not blob.endswith(b"\n") else b"")
        _, tab = coracle.digest_collapse(np.frombuffer(ref, dtype=np.uint8), dev.trim_params)
        table = D.CollapseTable(dev, min_keys=1 << 10)
        n = eng.digest_device(to_dev(dev, blob, pad), table, batch_bytes=batch)
        assert n == ref.count(b"\n") // 4, (case, pad, batch)
        assert table_dict(table) == tab.to_dict(), (case, pad, batch)


@pytest.mark.parametrize("world,cfg_id,tight", [(2, 1, False), (3, 2, False), (2, 2, True)])
def test_sharding_before_collapse_on_one_device_matches_oracle(dev, world, cfg_id, tight):
    """distributed.ShardedCollapse with ``world`` ranks on ONE device (loop-back instead of the all-to-all): every batch's
    insert list cut by owner (mirge_shard_scatter), the pieces placed at the end of the owners' arenas in source-rank
    order, key offsets rebased (mirge_shard_rebase), in-place insert -- everything of that path except NCCL -- against
    the single-process oracle.  ``tight``: regions far too small on the first try (the exact-size repeat of the scatter).
    (tests/test_gpu_multi.py runs the same with NCCL on two GPUs.)"""
    from mirge_b200 import device as D
    from mirge_b200 import distributed as MD
    from mirge_b200 import synth

    n_reads = 50_000
    libs = synth.make_libraries(scale=0.05, mrna_count=100)
    cfg = synth.trim_config_for(cfg_id)
    eng = D.DigestEngine(dev, cfg)
    fq = synth.ReadGenerator(libs, synth.CONFIGS[cfg_id], "cpu").fastq(n_reads).numpy()
    nl = np.flatnonzero(fq == 10)
    scs = [MD.ShardedCollapse(eng, world, overlap=False, slack=0.01 if tight else 1.2) for _ in range(world)]
    owners = [D.CollapseTable(dev, min_keys=1 << 12) for _ in range(world)]
    # unequal shards: rank 0 has several batches, the last rank a single one
    cuts = [0] + [int(n_reads * f) for f in ((0.6,) if world == 2 else (0.5, 0.85))] + [n_reads]
    shards = []
    for r in range(world):
        lo, hi = cuts[r], cuts[r + 1]
        b0 = 0 if lo == 0 else int(nl[4 * lo - 1]) + 1
        shards.append(torch.from_numpy(fq[b0 : int(nl[4 * hi - 1]) + 1].copy()).to(dev.tdev))
    pos = [0] * world
    batch = 2 << 20
    n_rec = 0
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
            cur = p["cursors"].cpu().numpy()
            if tight and br is not None and br.n_items > 5000:
                assert max(MD.ShardedCollapse.split_cursors(cur)[0]) > p["cap_items"]  # the first try did overflow
            p = scs[r].settle(p, cur)
            packed.append(p)
            sizes.append(MD.ShardedCollapse.split_cursors(p["cursors"].cpu().numpy()))
        for o in range(world):  # what the two all-to-alls deliver to owner o
            recv_it = [sizes[s][0][o] for s in range(world)]
            recv_w = [sizes[s][1][o] for s in range(world)]
            items, arena, bases = scs[o].place(owners[o], recv_it, recv_w)
            ai = aw = 0
            for s in range(world):
                ci, cw = packed[s]["cap_items"], packed[s]["cap_words"]
                items[ai : ai + recv_it[s]].copy_(packed[s]["items"][o * ci : o * ci + recv_it[s]])
                arena[aw : aw + recv_w[s]].copy_(packed[s]["keys"][o * cw : o * cw + recv_w[s]])
                ai += recv_it[s]
                aw += recv_w[s]
            scs[o].insert(owners[o], items, recv_it, bases)
    assert n_rec == n_reads
    union = {}
    for o in owners:
        d = table_dict(o)
        assert not (set(d) & set(union)), "a sequence is owned by two ranks"
        union.update(d)
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
    assert union == tab.to_dict()
    sizes = [o.n_keys for o in owners]
    assert min(sizes) > 0.6 * max(sizes), sizes  # the owner hash spreads the sequences evenly


@pytest.mark.parametrize("cfg_id", [1, 3])
def test_exchange_world2_on_one_device_matches_oracle(dev, cfg_id):
    """The multi-GPU exchange with world = 2 on ONE device (two local tables, two owner tables, loop-back transport):
    partition plan / totals / scatter, records received into the owners' arenas, mirge_collapse_merge_inplace --
    everything of the N > 1 path except NCCL -- against the single-process oracle.  (tests/test_gpu_multi.py runs the
    same with NCCL on two GPUs.)"""
    from mirge_b200 import device as D
    from mirge_b200 import distributed as MD
    from mirge_b200 import synth

    n_reads = 60_000
    libs = synth.make_libraries(scale=0.05, mrna_count=100)
    cfg = synth.trim_config_for(cfg_id)
    eng = D.DigestEngine(dev, cfg)
    umi = cfg.umi() or (0, 0)
    fq = synth.ReadGenerator(libs, synth.CONFIGS[cfg_id], "cpu").fastq(n_reads).numpy()
    nl = np.flatnonzero(fq == 10)
    locals_, pairs = [], []
    for lo, hi in MD.shard_ranges(n_reads, 2):
        b0 = 0 if lo == 0 else int(nl[4 * lo - 1]) + 1
        b1 = int(nl[4 * hi - 1]) + 1
        t = D.CollapseTable(dev, min_keys=1 << 12)
        assert eng.digest_device(torch.from_numpy(fq[b0:b1].copy()).to(dev.tdev), t, batch_bytes=3 << 20) == hi - lo
        locals_.append(t)
        pairs.append(t.drain())
    owners = [D.CollapseTable(dev, min_keys=1 << 12) for _ in range(2)]
    # two rounds of the same exchange: the second one meets every key again (merge into existing slots)
    for _ in range(2):
        MD.loopback_exchange([dev, dev], locals_, pairs, owners, umi=umi)
    union = {}
    for o in owners:
        d = table_dict(o)
        assert not (set(d) & set(union)), "a sequence is owned by two ranks"
        union.update(d)
    _, tab = coracle.digest_collapse(fq, dev.trim_params, nthreads=8)
    exp = tab.to_dict()
    if cfg.umi() is None:
        assert union == {k: 2 * v for k, v in exp.items()}
    else:
        # UMI mode partitions by the centre (flanks removed): both levels stay owner-local; first-level keys as such
        assert union == {k: 2 * v for k, v in exp.items()}
        centres = {}
        for i, o in enumerate(owners):
            keys = o.export_keys()
            for k in keys.tolist():
                c = k.decode()[umi[0] : len(k) - umi[1]] if umi[1] else k.decode()[umi[0] :]
                assert centres.setdefault(c, i) == i, "a centre sequence is split across owners"
