"""DuckDB-shaped LIST columns for the tests: per chunk a vector of duckdb_list_entry {uint64 offset, uint64 length},
a validity mask, and that chunk's own child vector (duckdb_list_vector_get_child / _get_size), the child vectors of
all chunks staged back to back (element child_base[k], mask words at child_val_off[k])."""
import numpy as np

from duckdb_mbt_b200 import chunks as ch


class ListColumn:
    pass


def make_list_column(n, width, pattern, seed, layout="contiguous", null_frac=0.2, child_null_frac=0.15, max_len=6):
    """layout: "contiguous" (entries in row order, back to back -- what a scan produces), "shuffled" (spans in a random
    order with gaps -- slices / selections), "shared" (rows may point at the same span)"""
    rng = np.random.default_rng(seed)
    counts = ch.chunk_counts(n, pattern, rng)
    nch = counts.shape[0]
    lc = ListColumn()
    lc.counts, lc.width = counts, width
    lc.valid = rng.random(n) >= null_frac if null_frac else np.ones(n, bool)
    lc.lens = rng.integers(0, max_len + 1, n).astype(np.uint64)
    entries = np.zeros((nch, ch.VECTOR_SIZE, 2), dtype=np.uint64)
    child_chunks, cmask_chunks, child_base, child_val_off, child_sizes = [], [], [], [], []
    lc.expected = []  # python lists (None = NULL row; None elements = NULL child)
    row, base_el, base_w = 0, 0, 0
    for k in range(nch):
        cnt = int(counts[k])
        lens = lc.lens[row: row + cnt]
        valid = lc.valid[row: row + cnt]
        if layout == "contiguous":
            starts = np.concatenate([[0], np.cumsum(np.where(valid, lens, 0))[:-1]]).astype(np.uint64) if cnt else np.zeros(0, np.uint64)
            size = int(np.where(valid, lens, 0).sum())
        else:
            order = rng.permutation(cnt)
            starts = np.zeros(cnt, np.uint64)
            pos = int(rng.integers(0, 3))
            for r in order:
                if layout == "shared" and pos > 8 and rng.random() < 0.3:
                    starts[r] = rng.integers(0, max(1, pos - int(lens[r])))
                else:
                    starts[r] = pos
                    pos += int(lens[r]) + int(rng.integers(0, 2))
            size = pos + 1
        vals = rng.integers(0, 256, (size, width), dtype=np.uint8)
        cvalid = rng.random(size) >= child_null_frac if child_null_frac else np.ones(size, bool)
        e = entries[k]
        e[:cnt, 0], e[:cnt, 1] = starts, lens
        # the entry of a NULL row is unspecified: garbage that must never be followed
        e[:cnt][~valid] = rng.integers(1 << 40, 1 << 50, (int((~valid).sum()), 2), dtype=np.uint64)
        for i in range(cnt):
            if not valid[i]:
                lc.expected.append(None)
            else:
                s, l = int(starts[i]), int(lens[i])
                lc.expected.append([bytes(vals[j]) if cvalid[j] else None for j in range(s, s + l)])
        words = np.zeros((size + 63) // 64 + 1, dtype=np.uint64)
        bits = np.packbits(cvalid.astype(np.uint8), bitorder="little")
        words.view(np.uint8)[: bits.shape[0]] = bits
        all_valid = bool(cvalid.all()) and k % 2 == 1  # some chunks hand out a NULL mask pointer
        child_chunks.append(vals.reshape(-1))
        child_base.append(base_el)
        child_sizes.append(size)
        child_val_off.append(-1 if all_valid else base_w)
        cmask_chunks.append(words)
        base_el += size
        base_w += words.shape[0]
        row += cnt
    lc.entries = entries.reshape(-1).view(np.uint8)
    lc.data_off = (np.arange(nch, dtype=np.uint64) * np.uint64(ch.VECTOR_SIZE * 16))
    lc.validity, lc.val_off = ch.make_validity(lc.valid if null_frac else None, counts, True)
    lc.child_data = np.concatenate(child_chunks) if child_chunks else np.zeros(0, np.uint8)
    lc.child_validity = np.concatenate(cmask_chunks) if cmask_chunks else np.zeros(1, np.uint64)
    lc.child_base = np.asarray(child_base, dtype=np.uint64)
    lc.child_val_off = np.asarray(child_val_off, dtype=np.int64)
    lc.child_sizes = np.asarray(child_sizes, dtype=np.uint64)
    lc.capacity = int(np.where(lc.valid, lc.lens, 0).sum())
    return lc


def as_column(lc, name, child_type, dec_width=0, dec_scale=0):
    """the LIST column as a chunks.Column for the host API (dmb_host_column + dmb_host_list)"""
    col = ch.Column(name, ch.T_LIST, ch.P_U128, lc.entries, lc.data_off, lc.validity, lc.val_off)
    col.list_child_type = child_type
    col.list_child_dec_width, col.list_child_dec_scale = dec_width, dec_scale
    col.list_child_data = lc.child_data
    col.list_child_base = lc.child_base
    col.list_child_sizes = lc.child_sizes
    col.list_child_validity = lc.child_validity
    col.list_child_val_off = lc.child_val_off
    return col


def as_described_column(lc, name, child_type):
    """the same LIST column with its child described as a column (dmb_host_list.child_col) instead of the flat fields"""
    col = ch.Column(name, ch.T_LIST, ch.P_U128, lc.entries, lc.data_off, lc.validity, lc.val_off)
    col.list_child_sizes = lc.child_sizes
    col.list_child_col = ch.Column("item", child_type, ch.phys_of_type(child_type), lc.child_data, lc.child_base * np.uint64(lc.width),
                                   lc.child_validity, lc.child_val_off)
    return col
