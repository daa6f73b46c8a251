"""Rank 0's side of the sharded SAM files (distributed.write_gathered_sam): records gathered from the owners land in
the per-round files in the single-process order -- file by file in round order (rounds 0 then 8 into one file), table
rows ascending, a sequence's records in its owner's order -- and records of sequences that are not a table row are
dropped.  Plain numpy; no GPU, no process group."""
import numpy as np

from mirge_b200 import distributed as MD


def owner_arrays(recs):
    """[bytes, lengths, key ids, rounds] of records given as (key id, round, text), in that order."""
    data = b"".join(t.encode() for _, _, t in recs)
    return [np.frombuffer(data, dtype=np.uint8).copy(), np.array([len(t) for _, _, t in recs], dtype=np.int64),
            np.array([k for k, _, _ in recs], dtype=np.int64), np.array([r for _, r, _ in recs], dtype=np.uint8)]


def test_records_land_in_table_order(tmp_path):
    # gathered key list: rank 0 owns keys 0..2 (global 0..2), rank 1 owns keys 0..3 (global 3..6)
    offs = np.array([0, 3, 7])
    # table rows in gathered order: row 0 = global 4, row 1 = global 0, row 2 = global 6, row 3 = global 2 (1, 3, 5 dropped)
    order = np.array([4, 0, 6, 2])
    g0 = owner_arrays([(0, 0, "k0.r0\n"), (1, 0, "dropped\n"), (2, 8, "k2.r8\n"), (0, 2, "k0.t1\n"), (0, 2, "k0.t0\n")])
    g1 = owner_arrays([(1, 0, "k4.r0\n"), (3, 0, "k6.r0\n"), (3, 2, "k6.t2\n"), (3, 2, "k6.t1\n"), (3, 2, "k6.t0\n"),
                       (0, 8, "dropped\n"), (1, 2, "k4.t0\n")])
    rounds = [(0, "miRge3_miRNA.sam"), (2, "miRge3_tRNA.sam"), (8, "miRge3_miRNA.sam")]
    n_rec, n_bytes = MD.write_gathered_sam(str(tmp_path), [g0, g1], rounds, order, offs, 7, batch=2)
    mir = (tmp_path / "miRge3_miRNA.sam").read_text()
    trna = (tmp_path / "miRge3_tRNA.sam").read_text()
    assert mir == "k4.r0\nk0.r0\nk6.r0\nk2.r8\n"
    assert trna == "k4.t0\nk0.t1\nk0.t0\nk6.t2\nk6.t1\nk6.t0\n"
    assert n_rec == 10 and n_bytes == len(mir) + len(trna)


def test_nothing_to_write_creates_no_file(tmp_path):
    empty = owner_arrays([])
    only_dropped = owner_arrays([(0, 3, "dropped\n")])
    no_rows = np.zeros(0, dtype=np.int64)  # (the one gathered key is no row of the table)
    n = MD.write_gathered_sam(str(tmp_path), [empty, only_dropped], [(3, "miRge3_pre_tRNA.sam")], no_rows, np.array([0, 0, 1]), 1)
    assert n == (0, 0) and not list(tmp_path.iterdir())
