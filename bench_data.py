"""Deterministic synthetic Parca-schema tables for bench.py and the full-size tests (SURVEY.md §8d).

Generator: u(k, i) = splitmix64(S ^ k*0x9E3779B97F4A7C15 ^ i), S = 0xF205DB.
  labels.l00 .. l{L-1}   optional RLE_DICTIONARY strings "v%06d" % (u(k,i) mod C_k), NULL when
                         u(100+k, i) mod 100 < p_k          (C = 64, 256, 16, 32, 8, 128, 4, 64, ...; p_k = 10 for k >= 2)
  example_type           "cpu"
  stacktrace             one of 4096 16-character ids
  timestamp              T0 + i      (int64, PLAIN)
  value                  u(200, i) mod 1000   (int64, PLAIN)
  floatvalue             (u(201, i) mod 10^6) / 1000.0   (optional double, PLAIN)
Rows are cut into parts of PART_ROWS rows; inside a part rows are sorted by the schema's sorting
columns (example_type, labels.*, timestamp, stacktrace; NULLs first) exactly as compaction leaves
them (samples/example.go:195-209, table.go:1296-1346), or left in arrival order with sort=False.
Each part is one Parquet file with row groups of RG_ROWS rows, written by pyarrow in FrostDB's
layout (frostdb_b200/dynparquet.py).
"""
from __future__ import annotations

import hashlib
import os
import tempfile
from concurrent.futures import ProcessPoolExecutor
from typing import Dict, List, Tuple

import numpy as np

from frostdb_b200 import dynparquet as dp

SEED = 0xF205DB
GOLD = 0x9E3779B97F4A7C15
T0 = 1_600_000_000_000
PART_ROWS = 4 * 1024 * 1024
RG_ROWS = 1024 * 1024
_CARD_CYCLE = [16, 32, 8, 128, 4, 64]


def cardinalities(n_labels: int, c0: int = 64, c1: int = 256) -> List[int]:
    out = []
    for k in range(n_labels):
        out.append(c0 if k == 0 else c1 if k == 1 else _CARD_CYCLE[(k - 2) % len(_CARD_CYCLE)])
    return out


def splitmix64(x: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        z = x + np.uint64(GOLD)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return z ^ (z >> np.uint64(31))


def u(k: int, i: np.ndarray) -> np.ndarray:
    with np.errstate(over="ignore"):
        return splitmix64(np.uint64(SEED) ^ np.uint64((k * GOLD) & 0xFFFFFFFFFFFFFFFF) ^ i)


def part_columns(first_row: int, n: int, n_labels: int, cards: List[int], *, sort: bool = True,
                 with_float: bool = False) -> Dict[str, object]:
    i = np.arange(first_row, first_row + n, dtype=np.uint64)
    labels = []
    for k in range(n_labels):
        idx = (u(k, i) % np.uint64(cards[k])).astype(np.int32)
        if k >= 2:
            idx[(u(100 + k, i) % np.uint64(100)) < np.uint64(10)] = -1
        labels.append(idx)
    stack = (u(300, i) % np.uint64(4096)).astype(np.int32)
    ts = (np.int64(T0) + i.astype(np.int64))
    value = (u(200, i) % np.uint64(1000)).astype(np.int64)
    fval = (u(201, i) % np.uint64(10**6)).astype(np.float64) / 1000.0 if with_float else None
    perm = None
    if sort:
        # pack (code = idx + 1, NULL = 0 sorts first) of l00.. into 64-bit words, most significant first
        words, cur, used = [], np.zeros(n, np.uint64), 0
        for k in range(n_labels):
            bits = int(cards[k]).bit_length()
            if used + bits > 64:
                words.append(cur << np.uint64(64 - used))
                cur, used = np.zeros(n, np.uint64), 0
            cur = (cur << np.uint64(bits)) | (labels[k] + 1).astype(np.uint64)
            used += bits
        if used:
            words.append(cur << np.uint64(64 - used))
        # timestamp ascending is the arrival order: a stable sort keeps it; stacktrace breaks no ties
        perm = np.lexsort(tuple(reversed(words))) if words else None
    def p(a):
        return a if perm is None else a[perm]
    cols: Dict[str, object] = {
        "example_type": (np.zeros(n, np.int32), ["cpu"]),
        "stacktrace": (p(stack), [f"{j:016x}" for j in range(4096)]),
        "timestamp": p(ts),
        "value": p(value),
    }
    for k in range(n_labels):
        cols[f"labels.l{k:02d}"] = (p(labels[k]), [f"v{j:06d}" for j in range(cards[k])])
    if with_float:
        cols["floatvalue"] = p(fval)
    return cols


def _write_part(args) -> Tuple[str, int]:
    path, first_row, n, n_labels, cards, sort, with_float, rg_rows = args
    schema = dp.SampleDefinitionWithFloat() if with_float else dp.SampleDefinition()
    cols = part_columns(first_row, n, n_labels, cards, sort=sort, with_float=with_float)
    buf = dp.write_part(schema, cols, sort=False, row_group_size=rg_rows)
    tmp = path + ".tmp"
    with open(tmp, "wb") as f:
        f.write(buf)
    os.replace(tmp, path)
    return path, len(buf)


def cache_dir(tag: str) -> str:
    """Where generated parts are kept between runs: in memory (/dev/shm) if possible, else the temporary directory.
    One directory per user, so that users sharing a machine never read or block each other's files."""
    for base in ("/dev/shm", tempfile.gettempdir()):
        if os.path.isdir(base) and os.access(base, os.W_OK):
            d = os.path.join(base, f"frostgpu_bench-{os.getuid()}", tag)
            os.makedirs(d, exist_ok=True)
            return d
    raise RuntimeError("no writable scratch directory")


def generate_parts(total_rows: int, n_labels: int, *, first_row: int = 0, sort: bool = True, with_float: bool = False,
                   part_rows: int = PART_ROWS, rg_rows: int = RG_ROWS, c0: int = 64, c1: int = 256,
                   workers: int = 0) -> List[str]:
    """Writes (or reuses) the part files of rows [first_row, first_row + total_rows) and returns their paths."""
    cards = cardinalities(n_labels, c0, c1)
    tag = hashlib.sha1(repr((SEED, total_rows, n_labels, first_row, sort, with_float, part_rows, rg_rows, cards, 3)).encode()).hexdigest()[:16]
    d = cache_dir(tag)
    jobs, paths = [], []
    r, pi = first_row, 0
    while r < first_row + total_rows:
        n = min(part_rows, first_row + total_rows - r)
        path = os.path.join(d, f"part_{pi:05d}.parquet")
        paths.append(path)
        if not os.path.exists(path):
            jobs.append((path, r, n, n_labels, cards, sort, with_float, rg_rows))
        r += n
        pi += 1
    if jobs:
        w = workers or min(len(jobs), max(1, (os.cpu_count() or 8) // 2), 32)
        if w <= 1:
            for j in jobs:
                _write_part(j)
        else:
            with ProcessPoolExecutor(max_workers=w) as ex:
                list(ex.map(_write_part, jobs))
    return paths
