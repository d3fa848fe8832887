"""ORACLE (test infrastructure): restatement of the decode kernels' rotated bin walk
(walk_start / scan_bin / segment_of in hpc-ops_b200/csrc/decode_common.cuh) over a task map read
back from a decode workspace, so tests can say which walks a launch took: where a walk starts inside
a task (that task is processed in two parts with the softmax state carried between them), which
bins straddle a kv-head boundary, and which short bins fall back to front to back.

Task-map ints: header int 0 = rows per bin + 1, int 1 = bins (CTAs), int 6 = tiles per kv head
(TB); bin i starts at row 1 + i * (int 0); a task row is ihead_kv, ibatch, ichunk, iseq_start,
num_seqkv, num_seqkvcache, num_tile_kv, num_tile_full, is_causal (12 ints); a row with int 0 or
int 1 negative ends the bin.
"""
from dataclasses import dataclass

import numpy as np

TASK_INTS = 12


@dataclass
class Walk:
    icta: int
    rows: np.ndarray  # [m, 12] valid task rows of the bin
    u0: int           # tile offset the rotation asks for (0: front to back)
    ks: int           # row the walk starts in
    o: int            # first tile of that row (0: the walk starts at a task boundary)

    @property
    def split(self):
        return self.o > 0

    @property
    def short(self):
        """Rotation asked for, but the bin has no tile at offset u0: walked front to back."""
        return self.u0 > 0 and int(self.rows[:, 6].sum()) <= self.u0

    @property
    def straddles_heads(self):
        return len(set(self.rows[:, 0].tolist())) > 1

    def segments(self):
        """[(row, first tile, end tile)] in processing order (the kernel's segment_of)."""
        m = len(self.rows)
        out = []
        for j in range(m + (1 if self.o > 0 else 0)):
            r = (self.ks + j) % m
            tb = self.o if j == 0 else 0
            te = self.o if j == m else int(self.rows[r, 6])
            out.append((r, tb, te))
        return out


def walk_start(task_map, icta):
    p = int(task_map[0]) - 1
    tb = int(task_map[6])
    if tb <= 0 or p <= 0:
        return 0
    c = ((icta * p) % tb) % p
    return (p - c) % p


def bin_rows(task_map, icta):
    ntpc1 = int(task_map[0])
    start = (1 + icta * ntpc1) * TASK_INTS
    rows = np.asarray(task_map[start:start + (ntpc1 - 1) * TASK_INTS]).reshape(-1, TASK_INTS)
    bad = np.nonzero((rows[:, 0] < 0) | (rows[:, 1] < 0))[0]
    return rows[:bad[0]] if len(bad) else rows


def scan_bin(rows, u0):
    """(ks, o): the row and tile the walk starts at; (0, 0) front to back or for a short bin."""
    if u0 <= 0:
        return 0, 0
    excl = 0
    for i, c in enumerate(rows[:, 6].tolist()):
        if excl <= u0 < excl + c:
            return i, u0 - excl
        excl += c
    return 0, 0


def walks(task_map, rotate=True):
    """Walk of every non-empty bin of a task map (int32 array, header first)."""
    task_map = np.asarray(task_map)
    out = []
    for icta in range(int(task_map[1])):
        rows = bin_rows(task_map, icta)
        if len(rows) == 0:
            continue
        u0 = walk_start(task_map, icta) if rotate else 0
        ks, o = scan_bin(rows, u0)
        out.append(Walk(icta, rows, u0, ks, o))
    return out


def tasks_of(task_map, ibatch, ihead_kv, rotate=True):
    """Describe the tasks of one (batch, kv head) pair: bin, row, chunk, key range, tiles, whether
    the rotated walk split it."""
    lines = []
    for w in walks(task_map, rotate):
        for r, row in enumerate(w.rows):
            if int(row[1]) == ibatch and int(row[0]) == ihead_kv:
                s = int(row[3])
                lines.append(f"bin {w.icta} row {r}: chunk {int(row[2])} keys [{s}, {s + int(row[4])})"
                             f" tiles {int(row[6])} causal {int(row[8])}"
                             + (f" split at tile {w.o}" if (w.split and r == w.ks) else ""))
    return "; ".join(lines)
