"""Multi-GPU collapse: one process per GPU (torch.distributed, NCCL over NVLink/NVSwitch).

The path shards naturally (SURVEY.md section 8e): FASTQ chunks / samples are split across ranks, every
rank collapses locally, and exactly one exchange makes each rank the owner of a disjoint slice of the
unique sequences: records (count, packed key) are partitioned by hash64(centre sequence) mod world
(kernel: mirge_partition_plan), packed per destination (mirge_partition_pack), moved with a single
all-to-all, and merged into the owner's table (mirge_collapse_merge).  With UMIs the centre (UMI flanks
removed) is hashed, so both UMI levels are owner-local.  Libraries are replicated; annotation then runs on
the owner's slice with no further communication.  The reference has no counterpart: its only
parallelism is a fork pool whose results are merged by one Python loop (digest.py:139-163)."""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import torch
import torch.distributed as dist


def shard_ranges(total: int, world: int):
    """Contiguous [lo, hi) unit ranges (chunks, samples, reads) per rank; sizes differ by at most 1."""
    base, rem = divmod(int(total), int(world))
    out, lo = [], 0
    for r in range(world):
        hi = lo + base + (1 if r < rem else 0)
        out.append((lo, hi))
        lo = hi
    return out


def gather_arrays(arrays, dst: int = 0, group=None, device=None):
    """Every rank's list of numpy arrays at rank ``dst``: returns [[arrays of rank 0], [arrays of rank 1], ...] there, None
    elsewhere.  The ranks pass the same number of arrays with the same dtype kinds; lengths (and, for byte strings, the
    item size) may differ.  One all-gather of the sizes, then one exact-size point-to-point transfer of raw bytes per
    rank -- no pickling of row objects (``gather_object``), which is what a cohort-sized table cannot afford.
    ``device``: where the transport wants its tensors (the rank's GPU for NCCL, None / cpu for gloo)."""
    import numpy as np

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    tdev = torch.device("cpu") if device is None else torch.device(device)
    glob = (lambda r: dist.get_global_rank(group, r)) if group is not None else (lambda r: r)
    arrs = [np.ascontiguousarray(a) for a in arrays]
    meta = torch.tensor([[a.size, a.dtype.itemsize] for a in arrs], dtype=torch.int64).reshape(-1).to(tdev)
    metas = [torch.empty_like(meta) for _ in range(world)]
    dist.all_gather(metas, meta, group=group)
    flat = np.concatenate([a.reshape(-1).view(np.uint8) for a in arrs]) if arrs else np.zeros(0, dtype=np.uint8)
    payload = torch.from_numpy(flat).to(tdev)
    if rank != dst:
        if payload.numel():
            dist.send(payload, glob(dst), group=group)
        return None
    out = []
    for r in range(world):
        sizes = metas[r].cpu().numpy().reshape(-1, 2)
        total = int((sizes[:, 0] * sizes[:, 1]).sum())
        if r == rank:
            raw = flat
        else:
            buf = torch.empty(total, dtype=torch.uint8, device=tdev)
            if total:
                dist.recv(buf, glob(r), group=group)
            raw = buf.cpu().numpy()
        got, o = [], 0
        for a, (n, item) in zip(arrs, sizes.tolist()):
            dt = np.dtype("S%d" % item) if a.dtype.kind == "S" else a.dtype
            if dt.itemsize != item:
                raise RuntimeError("gather_arrays: rank %d sent items of %d bytes where this rank has %s" % (r, item, a.dtype))
            got.append(raw[o : o + n * item].view(dt).reshape(n))
            o += n * item
        out.append(got)
    return out


def exchange_records(rec: torch.Tensor, sizes: torch.Tensor, send_recs: torch.Tensor, group=None,
                     send_words: torch.Tensor = None, recv_buffer=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """All-to-all of variable-size records.

    rec       int32 words of all records, grouped by destination rank (ascending)
    sizes     int32 [n] words of each record, same order
    send_recs int64 [world] number of records for each destination
    send_words optional int64 [world] words for each destination (computed from sizes when absent)
    recv_buffer optional callable (n_records, n_words) -> tensor the records are received into
    Returns (recv words, recv sizes) with records grouped by source rank.  Device-agnostic plumbing:
    NCCL on GPUs, gloo in the CPU tests."""
    world = dist.get_world_size(group)
    dev = rec.device
    send_recs = send_recs.to(torch.int64)
    if send_words is None:  # words per destination from the record sizes
        bounds = torch.zeros(world + 1, dtype=torch.int64, device=dev)
        bounds[1:] = torch.cumsum(send_recs.to(dev), 0)
        csum = torch.zeros(sizes.numel() + 1, dtype=torch.int64, device=dev)
        csum[1:] = torch.cumsum(sizes.to(torch.int64), 0)
        send_words = csum[bounds[1:]] - csum[bounds[:-1]]
    send_words = send_words.to(torch.int64).to(dev)
    meta_out = torch.stack([send_recs.to(dev), send_words]).t().contiguous()  # [world, 2]
    meta_in = torch.empty_like(meta_out)
    dist.all_to_all_single(meta_in, meta_out, group=group)
    meta_in_h = meta_in.cpu()
    recv_recs = [int(x) for x in meta_in_h[:, 0]]
    recv_words = [int(x) for x in meta_in_h[:, 1]]
    s_recs = [int(x) for x in send_recs.cpu()]
    s_words = [int(x) for x in send_words.cpu()]
    r_sizes = torch.empty(sum(recv_recs), dtype=sizes.dtype, device=dev)
    dist.all_to_all_single(r_sizes, sizes.contiguous(), output_split_sizes=recv_recs, input_split_sizes=s_recs, group=group)
    # recv_buffer(n_records, n_words) -> tensor of n_words elements to receive into (e.g. the end of a table's arena)
    r_rec = recv_buffer(sum(recv_recs), sum(recv_words)) if recv_buffer is not None else \
        torch.empty(sum(recv_words), dtype=rec.dtype, device=dev)
    dist.all_to_all_single(r_rec, rec.contiguous(), output_split_sizes=recv_words, input_split_sizes=s_words, group=group)
    return r_rec, r_sizes


def plan_and_pack(dev, local_table, ids: torch.Tensor, cnt: torch.Tensor, world: int, umi=(0, 0)):
    """Sender side of the exchange (every kernel through the C ABI): owner and record size of every drained
    (key id, count) pair -> totals per owner -> scatter into per-owner regions of one send buffer (cursors, no sort).
    Returns (rec int32 words grouped by owner, sizes int32 [n] in the same order, send_recs int64 [world],
    send_words int64 [world])."""
    from .device import _ptr

    lib = dev.lib
    n = int(ids.numel())
    if n > (1 << 16):
        # the drain lists the pairs in slot order, i.e. at random with respect to the arena; in key-id order (= creation
        # order = arena order) the two passes below stream the key text instead of chasing it (2.4 + 3.7 ms -> about a
        # third for 39 M keys)
        with dev.timed("xchg_order"):
            ids, order = torch.sort(ids)
            cnt = cnt[order]
            del order
    dest = dev.empty(n, torch.int32)
    words = dev.empty(n, torch.int32)
    totals = dev.zeros(2 * world, torch.int64)
    with dev.timed("xchg_plan"):
        if n:
            dev.check(lib.mirge_partition_plan(dev.ctx, C.byref(local_table.struct), _ptr(ids), n, int(umi[0]), int(umi[1]), world,
                                               _ptr(dest), _ptr(words), dev.stream()))
        dev.check(lib.mirge_partition_totals(dev.ctx, _ptr(dest), _ptr(words), n, world, _ptr(totals), dev.stream()))
        dev.launches += 2
        tot = totals.cpu()
    send_words, send_recs = tot[:world].clone(), tot[world:].clone()
    total = int(send_words.sum())
    if total >= (1 << 31):
        raise RuntimeError("exchange larger than 2^31 words per rank; lower the batch size")
    base = ((torch.cumsum(send_recs, 0) - send_recs) << 32) | (torch.cumsum(send_words, 0) - send_words)
    rec = dev.empty(total, torch.int32)
    sizes = dev.empty(n, torch.int32)
    with dev.timed("xchg_pack"):
        cursors = base.to(dev.tdev)
        if n:
            dev.check(lib.mirge_partition_scatter(dev.ctx, C.byref(local_table.struct), _ptr(ids), _ptr(cnt), _ptr(dest), _ptr(words), n,
                                                  world, _ptr(cursors), _ptr(rec), _ptr(sizes), dev.stream()))
            dev.launches += 1
    return rec[:total], sizes[:n], send_recs, send_words


def arena_receiver(owner_table):
    """(callable for exchange_records' recv_buffer, state): the records are received straight into the end of the
    owner's arena, where the first record of a sequence becomes the table's copy of its key (no copy, no fence)."""
    owner_table.check()
    state = {}

    def into_arena(n_rec, n_words):
        owner_table.reserve(n_rec, n_words)
        a0 = owner_table.arena_used
        state["a0"] = a0
        return owner_table.arena[a0 : a0 + n_words]

    return into_arena, state


def merge_received(dev, owner_table, r_rec: torch.Tensor, r_sizes: torch.Tensor, a0: int) -> int:
    """Owner side: the received records lie at arena word a0; merge them in place (mirge_collapse_merge_inplace)."""
    from .device import _ptr

    m = int(r_sizes.numel())
    if m == 0:
        return 0
    with dev.timed("xchg_merge"):
        r_off = (torch.cumsum(r_sizes.to(torch.int64), 0) - r_sizes.to(torch.int64) + a0)
        r_off = torch.where(r_off >= (1 << 31), r_off - (1 << 32), r_off).to(torch.int32)
        owner_table.arena_used = a0 + int(r_rec.numel())
        owner_table.ctrl[0:1].fill_(owner_table.arena_used)
        deferred = dev.empty(m, torch.int32)
        dev.check(dev.lib.mirge_collapse_merge_inplace(dev.ctx, C.byref(owner_table.struct), _ptr(r_off), m, _ptr(deferred), dev.stream()))
        dev.launches += 3
        owner_table.check()
    return m


def exchange_and_merge(dev, local_table, ids: torch.Tensor, cnt: torch.Tensor, owner_table, world: int, umi=(0, 0), group=None):
    """Partition the drained (key id, count) pairs of ``local_table`` by owner, exchange, merge into
    ``owner_table``: plan_and_pack -> all-to-all (received into the owner's arena) -> merge_received."""
    rec, sizes, send_recs, send_words = plan_and_pack(dev, local_table, ids, cnt, world, umi)
    into_arena, state = arena_receiver(owner_table)
    with dev.timed("xchg_a2a"):
        r_rec, r_sizes = exchange_records(rec, sizes, send_recs, group, send_words=send_words, recv_buffer=into_arena)
    return merge_received(dev, owner_table, r_rec, r_sizes, state.get("a0", 0))


def loopback_exchange(devs, local_tables, pairs, owner_tables, umi=(0, 0)):
    """The same exchange for ``world`` = len(local_tables) ranks that live in ONE process (tests on a single GPU, and
    single-process multi-table runs): every rank's send buffer is cut by owner and the pieces are copied into the
    owners' arenas in source-rank order -- what the all-to-all does -- then merged in place.  ``pairs[r]`` = (ids, cnt)
    drained from local_tables[r]; devs[r] = Device used for rank r's kernels."""
    world = len(local_tables)
    sent = [plan_and_pack(devs[r], local_tables[r], pairs[r][0], pairs[r][1], world, umi) for r in range(world)]
    merged = []
    for o in range(world):
        dev = devs[o]
        rec_parts, size_parts = [], []
        for r in range(world):
            rec, sizes, send_recs, send_words = sent[r]
            w0, r0 = int(send_words[:o].sum()), int(send_recs[:o].sum())
            rec_parts.append(rec[w0 : w0 + int(send_words[o])])
            size_parts.append(sizes[r0 : r0 + int(send_recs[o])])
        r_sizes = torch.cat(size_parts)
        n_words = sum(int(p.numel()) for p in rec_parts)
        into_arena, state = arena_receiver(owner_tables[o])
        dst = into_arena(int(r_sizes.numel()), n_words)
        at = 0
        for part in rec_parts:
            dst[at : at + part.numel()].copy_(part)
            at += int(part.numel())
        merged.append(merge_received(dev, owner_tables[o], dst, r_sizes, state["a0"]))
    return merged


class ShardedCollapse:
    """Collapse of ONE sample whose reads are spread over the ranks (bench.py weak scaling, a large sample cut by reads):
    sharding BEFORE the collapse.  Per batch of a rank's reads:

        pack      the batch's insert list (what the trim kernels wrote: packed keys + (key offset, count) items) is cut
                  by owner = hash(key) mod world into fixed-capacity regions (mirge_shard_scatter);
        sizes     one all-gather of the per-owner (items, words) tells every rank what it will receive; the flag that
                  rides along says whether the rank has more input, so ranks with fewer batches keep joining rounds;
        exchange  two all-to-alls with exact sizes (items; key words straight into the end of the owner's arena);
        insert    key offsets made absolute (mirge_shard_rebase), then the single-GPU collapse
                  (mirge_collapse_insert_list, keys in place).

    The rounds are software-pipelined: while round k is packed, round k - 1 is on the wire and round k - 2 is inserted.
    Collectives run on side streams (under the next batch's trim kernels; sizes and data on separate communicators, so
    a round's few bytes of sizes never queue behind the previous round's data) and the sizes come back through pinned
    memory: the launch stream never waits for the host or the network.  Every emitted key is inserted exactly once,
    into the table of the rank that owns it: there is no local table and no drain / sort / merge of unique sequences
    (exchange_and_merge above, still the path for samples dealt whole to ranks: baking_sharded).  Owner tables, key ids
    and the annotation that follows are the single-GPU ones.

        more = True
        for every local batch:  more = sc.round(table, br, has_more_input)
        sc.drain_rounds(table, more)          # join the other ranks' remaining rounds, insert the last arrivals
    """

    def __init__(self, eng, world: int, group=None, overlap: bool = True, slack: float = 1.2):
        self.eng, self.dev = eng, eng.dev
        self.world, self.group = int(world), group
        self.slack = float(slack)
        self.overlap = bool(overlap)
        self.size_group = group
        if group is None and dist.is_initialized() and dist.get_backend() == "nccl" and self.overlap:
            # The collectives run under the trim / collapse kernels of other rounds: NCCL's kernels must not queue behind
            # the CTAs of those grids, so this path gets its own communicators on high-priority streams -- two of them,
            # because a communicator runs its operations in order and the few bytes of a round's sizes must not wait for
            # the previous round's data (at 8 ranks that wait stalled the host once per round).  Collective: every rank
            # constructs its ShardedCollapse at the same point.
            try:
                opts = dist.ProcessGroupNCCL.Options()
                opts.is_high_priority_stream = True
                self.group = dist.new_group(backend="nccl", pg_options=opts)
                opts2 = dist.ProcessGroupNCCL.Options()
                opts2.is_high_priority_stream = True
                self.size_group = dist.new_group(backend="nccl", pg_options=opts2)
            except Exception:
                self.group = self.size_group = None
        # (the plumbing below also runs on a CPU device with the gloo backend -- no streams, events or pinned memory --
        # which is how tests/test_distributed_cpu.py drives the round protocol with stand-ins for the three kernels)
        self._cuda = self.dev.tdev.type == "cuda"
        self.comm = torch.cuda.Stream(device=self.dev.tdev, priority=-1) if self._cuda else None        # data: the two all-to-alls
        self.comm_sizes = torch.cuda.Stream(device=self.dev.tdev, priority=-1) if self._cuda else None  # sizes: all-gather + copy to the host
        self.q = []  # rounds in flight, oldest first
        self.rounds = 0
        self._pinned = []

    # -- sender ------------------------------------------------------------------------------------------------
    def pack(self, br, cap_items: int = 0, cap_words: int = 0):
        """Cut the batch's insert list by owner.  Returns a dict with the regions and their capacities."""
        from .device import _ptr

        d, W = self.dev, self.world
        n_items = int(br.n_items) if br is not None else 0
        words = int(br.arena_words) if br is not None else 0
        cap_items = max(int(cap_items), int(n_items / W * self.slack) + 1024)
        cap_words = max(int(cap_words), int(words / W * self.slack) + 8192)
        items = d.empty(W * cap_items, torch.int64)
        keys = d.empty(W * cap_words, torch.int32)
        cursors = d.empty(W, torch.int64)
        src_keys = None
        if n_items:
            if br.in_place:
                raise RuntimeError("ShardedCollapse.pack: the batch must be trimmed into a batch buffer (table=None)")
            src_keys = br.keys
        with d.timed("shard_pack"):
            d.check(d.lib.mirge_shard_scatter(d.ctx, _ptr(src_keys), _ptr(br.ins if n_items else None), n_items, W, cap_items, cap_words,
                                              _ptr(cursors), _ptr(items), _ptr(keys), d.stream()))
        d.launches += 1
        return {"items": items, "keys": keys, "cursors": cursors, "cap_items": cap_items, "cap_words": cap_words, "br": br}

    @staticmethod
    def split_cursors(cur):
        """(items[world], words[world]) from the packed cursors (host ints)."""
        return [int(c) >> 32 for c in cur], [int(c) & 0xFFFFFFFF for c in cur]

    def settle(self, packed, cur):
        """Repeat the scatter with exact capacities when a region was too small (skewed owners).  ``cur`` = this rank's
        cursors on the host; they are exact either way."""
        n_it, n_w = self.split_cursors(cur)
        if max(n_it) <= packed["cap_items"] and max(n_w) <= packed["cap_words"]:
            return packed
        return self.pack(packed["br"], max(n_it) + 1, max(n_w) + 1)

    def _gather_sizes(self, packed, more: bool):
        """All-gather of the cursors (+ the 'more input' flag) on the side stream, result on its way to pinned memory."""
        W = self.world
        if not self._cuda:
            mine = torch.empty(W + 1, dtype=torch.int64)
            mine[:W] = packed["cursors"]
            mine[W] = 1 if more else 0
            parts = [torch.empty(W + 1, dtype=torch.int64) for _ in range(W)]
            dist.all_gather(parts, mine, group=self.size_group)
            return torch.stack(parts), None
        main = torch.cuda.current_stream(self.dev.tdev)
        host = self._pinned.pop() if self._pinned else torch.empty((W, W + 1), dtype=torch.int64).pin_memory()
        cs = self.comm_sizes
        cs.wait_stream(main)
        packed["cursors"].record_stream(cs)
        with torch.cuda.stream(cs):
            mine = torch.empty(W + 1, dtype=torch.int64, device=self.dev.tdev)
            mine[:W] = packed["cursors"]
            mine[W:].fill_(1 if more else 0)  # (a kernel argument; ``mine[W] = ...`` is a pageable copy that blocks the host)
            allc = torch.empty((W, W + 1), dtype=torch.int64, device=self.dev.tdev)
            dist.all_gather_into_tensor(allc.view(-1), mine, group=self.size_group)
            host.copy_(allc, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(cs)
        return host, ev

    # -- receiver ----------------------------------------------------------------------------------------------
    def place(self, table, recv_items, recv_words):
        """Room for the received keys at the end of the owner's arena: (items buffer, arena slice, key bases)."""
        d = self.dev
        n_it, n_w = int(sum(recv_items)), int(sum(recv_words))
        if table.arena_used + n_w > table.arena.numel() and self.comm is not None:
            self.comm.synchronize()  # the arena is about to move: nothing may still be arriving in the old one
        table.reserve(n_it, n_w)
        a0 = table.arena_used
        bases, at = [], a0
        for w in recv_words:
            bases.append(at)
            at += int(w)
        table.arena_used = at
        table.ctrl[0:1].fill_(at)
        return d.empty(n_it, torch.int64), table.arena[a0:at], bases

    def insert(self, table, items, recv_items, bases, local_br=None):
        """The received items into the owner's table (keys already in its arena)."""
        import ctypes as C

        from .device import _ptr

        d, W = self.dev, self.world
        st_ = self.eng.stats
        if local_br is not None:  # the rank's own reads: what bench.py's rooflines are quoted on
            st_["records"] += local_br.n_records
            st_["bytes"] += local_br.consumed
            st_["emitted"] += local_br.n_emitted
            st_["key_words"] += local_br.key_words
        n = int(sum(recv_items))
        if n == 0:
            return
        cnt = (C.c_uint64 * W)(*[int(x) for x in recv_items])
        kb = (C.c_uint64 * W)(*[int(x) for x in bases])
        with d.timed("shard_rebase"):
            d.check(d.lib.mirge_shard_rebase(d.ctx, _ptr(items), W, cnt, kb, d.stream()))
        table.reserve(n, 0)
        scratch = d.empty(2 * n, torch.int32)
        with d.timed("collapse"):
            d.check(d.lib.mirge_collapse_insert_list(d.ctx, C.byref(table.struct), _ptr(table.arena), _ptr(items), n, _ptr(scratch), d.stream()))
        d.launches += 5
        before = table.n_keys
        table.check()
        table.new_frac = (table.n_keys - before) / max(n, 1)

    # -- the pipeline (collective) -----------------------------------------------------------------------------------
    def _exchange(self, table, r) -> bool:
        """Stage 2 of round r: its sizes have arrived -> room in the arena, the two all-to-alls on the side stream.
        Returns whether any rank announced more input in that round."""
        W = self.world
        rank = dist.get_rank(self.group)
        main = torch.cuda.current_stream(self.dev.tdev) if self._cuda else None
        if r["ev_sizes"] is not None:
            r["ev_sizes"].synchronize()
        allc = r["host"].numpy().copy()
        if self._cuda:
            self._pinned.append(r["host"])
        r.pop("host")
        packed = r["packed"]
        again = self.settle(packed, allc[rank, :W])
        if again is not packed:
            packed = r["packed"] = again
            if self._cuda:
                self.comm.wait_stream(main)  # (the repeated scatter runs on the launch stream)
        send_it, send_w = self.split_cursors(allc[rank, :W])
        recv_it, recv_w = [int(allc[s, rank]) >> 32 for s in range(W)], [int(allc[s, rank]) & 0xFFFFFFFF for s in range(W)]
        r_items, r_keys, bases = self.place(table, recv_it, recv_w)
        ci, cw = packed["cap_items"], packed["cap_words"]
        s_items = [packed["items"][d * ci : d * ci + send_it[d]] for d in range(W)]
        s_keys = [packed["keys"][d * cw : d * cw + send_w[d]] for d in range(W)]
        o_items = list(torch.split(r_items, recv_it)) if r_items.numel() else [r_items[:0]] * W
        o_keys = list(torch.split(r_keys, recv_w)) if r_keys.numel() else [r_keys[:0]] * W
        def wire():
            # what this rank owns itself does not go through the communicator: a device-to-device copy
            o_items[rank].copy_(s_items[rank], non_blocking=True)
            o_keys[rank].copy_(s_keys[rank], non_blocking=True)
            o_items[rank], s_items[rank] = r_items[:0], packed["items"][:0]
            o_keys[rank], s_keys[rank] = r_keys[:0], packed["keys"][:0]
            if W > 1:
                self._all_to_all(o_items, s_items)
                self._all_to_all(o_keys, s_keys)

        ev = None
        if self._cuda:
            for t in (packed["items"], packed["keys"], r_items, table.arena):
                t.record_stream(self.comm)
            with torch.cuda.stream(self.comm):
                with self.dev.timed("shard_a2a"):
                    wire()
                ev = torch.cuda.Event()
                ev.record(self.comm)
        else:
            wire()
        r.update(items=r_items, recv_items=recv_it, bases=bases, ev_data=ev, stage=2)
        return bool(allc[:, W].any())

    def _all_to_all(self, outs, ins):
        """Exact-size all-to-all of per-peer tensors (NCCL: grouped send / receive; gloo has no list form, the CPU tests
        go through point-to-point operations)."""
        if self._cuda:
            dist.all_to_all(outs, ins, group=self.group)
            return
        rank = dist.get_rank(self.group)
        reqs = []
        for peer in range(self.world):
            if peer == rank:
                continue
            if ins[peer].numel():
                reqs.append(dist.isend(ins[peer].contiguous(), peer, group=self.group))
            if outs[peer].numel():
                reqs.append(dist.irecv(outs[peer], peer, group=self.group))
        for q in reqs:
            q.wait()

    def _insert_round(self, table, r, on_piece=None):
        if r["ev_data"] is not None:
            torch.cuda.current_stream(self.dev.tdev).wait_event(r["ev_data"])
        self.insert(table, r["items"], r["recv_items"], r["bases"], r["packed"]["br"])
        if on_piece is not None:
            on_piece(table)

    def round(self, table, br, more: bool, on_piece=None) -> bool:
        """One collective round: this rank's batch ``br`` (None: no input left; ``more``: whether input remains after it)
        is packed and its sizes announced; the previous round goes on the wire; the one before is inserted
        (``on_piece(table)`` after it).  Returns False once every rank's input is known to be exhausted -- nothing was
        announced then and the caller must stop calling (drain_rounds does the rest); True otherwise.

        Every hand-over has a round of slack: the sizes announced in round k are read in round k + 1 (after that batch's
        trim), the data put on the wire in round k + 1 is waited for -- by the launch stream, not the host -- in round
        k + 2.  (Reading the sizes in the round that announces them would make every round a barrier between the
        ranks.)"""
        packed = self.pack(br)  # (first: the scatter follows the trim kernels without waiting for the host work below)
        any_more = True
        if self.q and self.q[-1]["stage"] == 1:
            any_more = self._exchange(table, self.q[-1])
        if not any_more:
            if br is not None and br.n_records:
                raise RuntimeError("ShardedCollapse: a batch arrived after every rank had announced the end of its input")
            return False
        host, ev = self._gather_sizes(packed, more)
        self.q.append({"stage": 1, "packed": packed, "host": host, "ev_sizes": ev})
        self.rounds += 1
        depth = 2 if self.overlap else 0
        while len(self.q) > depth and self.q[0]["stage"] == 2:
            self._insert_round(table, self.q.pop(0), on_piece)
        if not self.overlap:  # in line: exchange and insert this round now
            any_more = self._exchange(table, self.q[-1])
            self._insert_round(table, self.q.pop(0), on_piece)
            return any_more
        return True

    def drain_rounds(self, table, more_any: bool = True, on_piece=None):
        """After a rank's last batch: keep joining rounds while another rank may have input, then insert what is still
        on its way.  Leaves the object ready for the next sample."""
        while more_any:
            more_any = self.round(table, None, False, on_piece)
        while self.q:
            r = self.q.pop(0)
            if r["stage"] == 1:  # (cannot happen after a False round; kept for symmetry)
                self._exchange(table, r)
            self._insert_round(table, r, on_piece)

    def digest_device(self, buf: torch.Tensor, table, batch_bytes: int = 256 << 20, on_piece=None) -> int:
        """DigestEngine.digest_device for a rank's shard of the sample: returns the records this rank parsed; ``table``
        ends up holding the keys this rank owns with their counts over ALL ranks' reads."""
        from .device import FastqFormatError

        eng = self.eng
        total, pos, n_records = int(buf.numel()), 0, 0
        more_any = True
        while pos < total:
            end = min(total, pos + batch_bytes)
            final = end == total
            br = eng.trim_batch(buf[pos:end], end - pos, final, keep=False, table=None)
            if br.consumed == 0 and not final:
                raise FastqFormatError("no complete FASTQ record in batch")
            pos += br.consumed if not final else (end - pos)
            n_records += br.n_records
            more_any = self.round(table, br, pos < total, on_piece)
        self.drain_rounds(table, more_any, on_piece)
        return n_records


class ExchangeWorker:
    """The exchange off the critical path.  ``exchange_and_merge`` is a chain of small kernels, three collectives and
    host round trips for their split sizes (about 12 ms per 50 M-read pass, during which the trim kernels of the next
    batch could run).  A worker thread drives it on its own CUDA stream -- and with its own library context, whose
    pinned staging words the *_sync calls of the main thread must not share -- in submission order, which is the same
    on every rank, so the collectives line up.  The caller digests batch k + 1 into a second local table meanwhile and
    waits for the hand-over of batch k before it reuses that table.

        w = ExchangeWorker(device_index, owner_min_keys, world)
        h = w.submit(local_table, ids, cnt)        # after local_table.drain() on the main stream
        ...                                        # next batch, other local table
        h.wait()                                   # before local_table.reset()
        owner = w.finish()                         # all merges done; the owner table belongs to the caller again
    """

    class Handle:
        def __init__(self):
            import threading

            self._ev = threading.Event()
            self.result = None
            self.error = None

        def wait(self):
            self._ev.wait()
            if self.error is not None:
                raise self.error
            return self.result

    def __init__(self, index: int, world: int, owner_min_keys: int = 1 << 22, umi=(0, 0), group=None):
        import queue
        import threading

        from .device import CollapseTable, Device

        self.dev = Device(index)  # own context: own pinned staging for the synchronising calls
        self.owner = CollapseTable(self.dev, min_keys=owner_min_keys)
        self.world, self.umi, self.group = world, umi, group
        self.stream = torch.cuda.Stream(device=self.dev.tdev)
        self.q = queue.Queue()
        self.thread = threading.Thread(target=self._run, name="mirge-exchange", daemon=True)
        self.thread.start()

    def _run(self):
        torch.cuda.set_device(self.dev.tdev)
        with torch.cuda.stream(self.stream):
            while True:
                item = self.q.get()
                if item is None:
                    return
                kind, h, args = item
                try:
                    if kind == "xchg":
                        table, ids, cnt, ev, drain = args
                        self.stream.wait_event(ev)
                        ids.record_stream(self.stream)
                        cnt.record_stream(self.stream)
                        exchange_and_merge(self.dev, table, ids, cnt, self.owner, self.world, self.umi, self.group)
                        h.result = self.owner.drain() if drain else None
                    elif kind == "reset":
                        self.owner.reset()
                    self.stream.synchronize()
                except BaseException as exc:  # surfaces in wait()
                    h.error = exc
                h._ev.set()

    def submit(self, local_table, ids: torch.Tensor, cnt: torch.Tensor, drain_owner: bool = False) -> "ExchangeWorker.Handle":
        """Queue the exchange of the pairs drained from ``local_table`` (collective: every rank submits the same
        sequence of calls).  With ``drain_owner`` the handle's result is ``owner.drain()`` after the merge."""
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev.tdev))
        h = ExchangeWorker.Handle()
        self.q.put(("xchg", h, (local_table, ids, cnt, ev, drain_owner)))
        return h

    def reset_owner(self) -> "ExchangeWorker.Handle":
        h = ExchangeWorker.Handle()
        self.q.put(("reset", h, None))
        return h

    def finish(self):
        """Block until everything queued has run; the current stream then sees the owner table's final state."""
        h = ExchangeWorker.Handle()
        self.q.put(("noop", h, None))
        h.wait()
        return self.owner

    def close(self):
        self.q.put(None)
        self.thread.join()


# ---------------------------------------------------------------------------------------------------
# The two entry points for one process per GPU (torchrun): same arguments and, on rank 0, the same return
# values as digest.baking / manifoldAlign.bwtAlign.  Samples are dealt round-robin to the ranks (a sample's
# reads -- and with UMIs its first-level table -- stay on one GPU), every sample's unique sequences are
# hash-partitioned to their owners with one all-to-all, owners keep the per-sample counts of their slice and
# annotate it against replicated libraries; rank 0 gathers (sequence, counts, annotation) for the DataFrame
# (SURVEY.md section 8e).
# ---------------------------------------------------------------------------------------------------

_SHARD = {}


def assemble_table(gathered, names):
    """The sample x sequence DataFrame of ``baking`` (digest.py:237-261: outer join = sorted union of the sequences, 0
    where a sample lacks one, annotation columns empty, annotFlag 0) from what the owners sent: per rank
    (keys 'S' array, [(ids, counts) per sample]) with ids indexing that rank's keys.  Returns (df, order, offs, n_all):
    ``order`` = rows of the concatenated key list in table order (keys no sample counted are dropped), ``offs`` = first
    row of every rank in that list."""
    import numpy as np
    import pandas as pd

    from . import digest as DG

    sizes = [int(g[0].shape[0]) for g in gathered]
    offs = np.concatenate([[0], np.cumsum(sizes)])
    width = max([g[0].dtype.itemsize for g in gathered] + [1])
    all_keys = np.concatenate([g[0].astype("S%d" % width) for g in gathered]) if sum(sizes) else np.zeros(0, dtype="S1")
    mat = np.zeros((all_keys.shape[0], len(names)), dtype=np.int64)
    for r, (_, ps) in enumerate(gathered):
        for j, (i_, c_) in enumerate(ps):
            mat[offs[r] + i_, j] = c_
    seen = mat.any(axis=1) if mat.size else np.zeros(0, dtype=bool)
    order = np.argsort(all_keys, kind="stable")
    order = order[seen[order]]
    # frame built as digest.build_matrix builds it: beyond ARROW_INDEX_MIN rows no Python object per cell
    m = int(order.shape[0])
    index = DG.sequence_index(all_keys[order]) if m else pd.Index([], name="Sequence", dtype=object)
    frame = {"annotFlag": np.zeros(m, dtype=np.dtype(int))}
    empty = DG.empty_flag_column(m)
    frame.update((f, empty) for f in DG.INITIAL_FLAGS)
    df = pd.DataFrame(frame, index=index, copy=False)
    for j, name in enumerate(names):
        df[name] = mat[order, j]
    return df, order, offs, int(all_keys.shape[0])


def baking_sharded(args, inFileArray, inFileBaseArray, workDir, device=None, count_mode=None, batch_bytes=256 << 20, group=None):
    """Call on every rank.  Returns (complete_set, sampleReadCounts, trimmedReadCounts, trimmedReadCountsUnique);
    complete_set is the DataFrame of digest.baking on rank 0 and None elsewhere."""
    import numpy as np

    from . import digest as DG
    from . import params as P
    from .device import CollapseTable, Device, DigestEngine

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    cfg = P.TrimConfig.from_args(args, count_mode or DG.default_count_mode())
    dev = device or Device(torch.cuda.current_device())
    eng = DigestEngine(dev, cfg)
    umi = cfg.umi()
    local = CollapseTable(dev, min_keys=1 << 20)
    first_level = CollapseTable(dev, min_keys=1 << 20) if umi is not None else None
    owner = CollapseTable(dev, min_keys=1 << 20)
    streamer = DG.HostStreamer(eng, batch_bytes)
    names = list(inFileBaseArray)
    counts_read = np.zeros(len(names), dtype=np.int64)
    per_sample = []  # (owner ids, counts) of this rank's slice, per sample
    empty = torch.zeros(0, dtype=torch.int32, device=dev.tdev)
    # this rank's files are read / inflated ahead of the sample it is digesting (ingest.py)
    mine = [s for s in range(len(inFileArray)) if s % world == rank]
    readahead = DG.ingest.SampleReadahead([str(inFileArray[s]) for s in mine], threads=DG._host_threads(args))
    for s, path in enumerate(inFileArray):
        if s % world == rank:
            umi_csv = None
            if umi is not None and getattr(args, "umiDedup", False):
                import os

                umi_csv = os.path.join(str(workDir), names[s] + "_umiCounts.csv")
            with readahead.open(mine.index(s)) as f:
                res = DG.digest_sample(eng, f, local, first_level, bool(getattr(args, "umiDedup", False)), batch_bytes, umi_csv, streamer)
            counts_read[s] = res.count
            if getattr(args, "tcf_out", False):
                # <sample>.trim.collapse.fa (digest.py:226-235) by the rank that digested the sample: its local table
                # holds exactly the sample's completeDict
                DG.write_tcf(workDir, names[s], local, res)
            ids, cnt = res.ids_d, res.counts_d
        else:
            ids, cnt = empty, empty
        exchange_and_merge(dev, local, ids, cnt, owner, world, group=group)  # collective
        o_ids, o_cnt = owner.drain()
        per_sample.append((o_ids.cpu().numpy().astype(np.int64), o_cnt.cpu().numpy().astype(np.int64)))
        local.reset()
    readahead.close()
    # counters (digest.py:212-217): records parsed by the digesting rank, emitted counts and unique sequences
    # summed over the owners
    tot = torch.zeros((3, len(names)), dtype=torch.int64, device=dev.tdev)
    tot[0] = torch.from_numpy(counts_read).to(dev.tdev)
    tot[1] = torch.tensor([int(c.sum()) for _, c in per_sample], dtype=torch.int64, device=dev.tdev)
    tot[2] = torch.tensor([int(i.size) for i, _ in per_sample], dtype=torch.int64, device=dev.tdev)
    dist.all_reduce(tot, group=group)
    tot_h = tot.cpu().numpy()
    src = {n: int(tot_h[0, j]) for j, n in enumerate(names)}
    trc = {n: int(tot_h[1, j]) for j, n in enumerate(names)}
    tru = {n: int(tot_h[2, j]) for j, n in enumerate(names)}
    keys = owner.export_keys()
    # the owners' keys and per-sample (id, count) columns at rank 0 as raw arrays (no pickled rows)
    flat = gather_arrays([keys] + [a for pair in per_sample for a in pair], 0, group, dev.tdev if "nccl" in str(dist.get_backend(group)) else None)
    gathered = None if flat is None else [(g[0], [(g[1 + 2 * j], g[2 + 2 * j]) for j in range(len(names))]) for g in flat]
    _SHARD.clear()
    _SHARD.update(dev=dev, owner=owner, n_own=int(keys.shape[0]))
    if rank != 0:
        return None, src, trc, tru
    df, order, offs, n_all = assemble_table(gathered, names)
    _SHARD.update(order=order, offs=offs, n_all=n_all)
    # index_data.js read-length histograms (digest.py:270-295) from the gathered matrix; the UMI count histograms stay
    # with the single-process baking (their per-sample lists live on the digesting ranks)
    class _NoHist:
        hist = np.zeros(0, dtype=np.int64)

    DG._write_histograms(workDir, df, [_NoHist()] * len(names), names, None)
    return df, src, trc, tru


def fill_annotation(pdDataFrame, annot_all, ref_all, order, names_of, spike: bool):
    """What ``bwtAlign`` leaves in the table (manifoldAlign.py:50-56,137-141) from the owners' results: ``annot_all`` /
    ``ref_all`` = round (0xFF: none) and reference index of every gathered sequence in gather order, ``order`` = the
    table's rows in that order (assemble_table), ``names_of[round]`` = the reference names of the round's library.
    The round's column gets the reference name, annotFlag 1; the spike-in column goes unless ``-spk``."""
    import numpy as np

    a, ref = annot_all[order], ref_all[order]
    colnames = list(pdDataFrame.columns)
    for rnd in range(10 if spike else 9):
        rows = np.nonzero(a == rnd)[0]
        if rows.size == 0:
            continue
        col = pdDataFrame[colnames[1 + rnd]].to_numpy(dtype=object, copy=True)
        col[rows] = np.asarray(names_of[rnd], dtype=object)[ref[rows]]
        pdDataFrame[colnames[1 + rnd]] = col
    flag = pdDataFrame[colnames[0]].to_numpy(copy=True)
    flag[a != 0xFF] = 1
    pdDataFrame[colnames[0]] = flag
    if not spike:
        pdDataFrame = pdDataFrame.drop(columns=["spike-in"])
    return pdDataFrame.fillna("")


def owner_sam_records(dev, libs, keys, annot, hit_d, rounds):
    """The SAM records of the sequences a rank owns for the (round, file) pairs ``rounds`` (manifoldAlign.sam_rounds),
    formatted on its GPU: [record bytes uint8, record lengths int64, owner key id int64, round uint8], records grouped
    by round, key ids ascending inside a round and, inside a sequence, in the order bowtie prints them."""
    import numpy as np

    from . import manifoldAlign as MA
    from .libraries import ROUND_LIBS, round_policies

    pols = round_policies()
    data, lens, ids, rnds = [], [], [], []
    for rnd, _ in rounds:
        own = np.nonzero(annot == rnd)[0]
        if own.size == 0:
            continue
        lib = libs[ROUND_LIBS[rnd]]
        rec_ids, rec_hits = MA.round_sam_pairs(dev, lib, pols[rnd], keys, own, hit_d)
        for chunk, n in MA.sam_records(dev, lib, pols[rnd], keys, rec_ids, rec_hits):
            data.append(chunk)
            lens.append(n)
        ids.append(rec_ids)
        rnds.append(np.full(rec_ids.size, rnd, dtype=np.uint8))
    cat = lambda parts, dt: np.concatenate(parts).astype(dt, copy=False) if parts else np.zeros(0, dtype=dt)
    return [cat(data, np.uint8), cat(lens, np.int64), cat(ids, np.int64), cat(rnds, np.uint8)]


def write_gathered_sam(workDir, gathered, rounds, order, offs, n_all, batch: int = 1 << 20):
    """Rank 0: the owners' SAM records (per rank, what owner_sam_records returned) appended to the per-round files in the
    order the single-process bwtAlign writes them: file by file in round order, table rows ascending, a sequence's
    records in their owner's order.  Records of sequences that are not a row of the table (no sample counted them,
    assemble_table) are dropped.  Returns (records, bytes) written."""
    import os

    import numpy as np

    row_of = np.full(n_all, -1, dtype=np.int64)
    row_of[order] = np.arange(order.size, dtype=np.int64)
    data = np.concatenate([g[0] for g in gathered])
    lens = np.concatenate([g[1] for g in gathered])
    rows = np.concatenate([row_of[offs[r] + g[2]] for r, g in enumerate(gathered)])
    rnds = np.concatenate([g[3] for g in gathered])
    start = np.cumsum(lens) - lens
    n_rec = n_bytes = 0
    for rnd, fname in rounds:
        sel = np.nonzero((rnds == rnd) & (rows >= 0))[0]
        if sel.size == 0:
            continue
        sel = sel[np.argsort(rows[sel], kind="stable")]
        with open(os.path.join(str(workDir), fname), "ab") as fh:
            for b in range(0, sel.size, batch):
                s = sel[b : b + batch]
                ln = lens[s]
                at = np.cumsum(ln) - ln
                src = np.repeat(start[s] - at, ln) + np.arange(int(ln.sum()), dtype=np.int64)
                fh.write(memoryview(data[src]))
                n_bytes += int(ln.sum())
        n_rec += int(sel.size)
    return n_rec, n_bytes


def bwtAlign_sharded(args, pdDataFrame, workDir, ref_db, libraries=None, group=None):
    """Call on every rank after baking_sharded (pdDataFrame: its result on rank 0, None elsewhere).  Every rank
    annotates the sequences it owns; rank 0 returns the DataFrame manifoldAlign.bwtAlign would return.  With -bam /
    -trf every rank formats the SAM records of its own sequences and rank 0 writes the per-round files, the same bytes
    the single-process bwtAlign writes; the other ranks write nothing."""
    import numpy as np

    from . import manifoldAlign as MA
    from .libraries import ROUND_LIBS

    rank, world = dist.get_rank(group), dist.get_world_size(group)
    dev, owner = _SHARD["dev"], _SHARD["owner"]
    libs = libraries or MA.load_libraries(args, ref_db, dev)
    spike = bool(getattr(args, "spikeIn", False))
    keys = MA.KeySet.from_table(owner)
    annot_d, hit_d = MA.annotate_keys(dev, libs, keys, spike)
    annot = annot_d.cpu().numpy()
    _, _mm, ref, _off = MA.decode_hits(annot, hit_d.cpu().numpy())
    # round and reference index of every owned sequence at rank 0; the names are looked up there (libraries are replicated)
    tdev = dev.tdev if "nccl" in str(dist.get_backend(group)) else None
    gathered = gather_arrays([annot.astype(np.uint8), ref.astype(np.int64)], 0, group, tdev)
    rounds = MA.sam_rounds(args, spike)
    sam = gather_arrays(owner_sam_records(dev, libs, keys, annot, hit_d, rounds), 0, group, tdev) if rounds else None
    if rank != 0:
        return None
    if _SHARD["n_all"]:
        annot_all = np.concatenate([g[0] for g in gathered])
        ref_all = np.concatenate([g[1] for g in gathered])
    else:
        annot_all, ref_all = np.zeros(0, dtype=np.uint8), np.zeros(0, dtype=np.int64)
    if sam is not None:
        write_gathered_sam(workDir, sam, rounds, _SHARD["order"], _SHARD["offs"], _SHARD["n_all"])
    names_of = {rnd: libs[ROUND_LIBS[rnd]].names for rnd in range(10 if spike else 9)}
    return fill_annotation(pdDataFrame, annot_all, ref_all, _SHARD["order"], names_of, spike)
