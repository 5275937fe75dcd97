"""Ragged count matrices for the per-element data-term tests (tests/test_gpu_ragged.py, tests/test_oracle_ragged.py).

Every case is a full matrix whose every column is populated (so the column scales are finite) and one batch cut
from it at a nonzero row offset, so that the batch's row pointers start at a nonzero global offset.  The batches
carry the structure sparse kernels branch on: empty rows and columns, every row length against every alignment,
columns that span or end exactly on the column pass's 256-entry slices, rows longer than the hot split's
2048-entry stash, counts on either side of the lgamma table and of the compact upload formats, and batch sizes
one past a 128-row tile.  Every case has at least 64 columns populated in more than 5 % of its rows, so a model
with hot_density=0.05 has a tensor-core block of hot columns (and, but for `empty_cols`, cold columns too).
"""
from dataclasses import dataclass

import numpy as np


@dataclass
class Case:
    name: str
    x: np.ndarray            # full (N, D) float32 matrix, every column populated
    start: int               # first row of the batch
    B: int                   # rows of the batch

    @property
    def batch(self):
        return self.x[self.start:self.start + self.B]

    @property
    def D(self):
        return self.x.shape[1]


def _sparse(rng, B, D, hot=96, p_hot=0.3, p_cold=0.01, hi=6):
    """Counts with a dense-ish block of `hot` columns and a sparse remainder."""
    p = np.full(D, p_cold)
    p[:hot] = p_hot
    mask = rng.random((B, D)) < p[None, :]
    return np.where(mask, rng.integers(1, hi, size=(B, D)), 0).astype(np.float32)


def _frame(rng, batch, pre, post=4):
    """`pre` rows before and `post` rows after the batch; the rows after it populate every column."""
    B, D = batch.shape
    x = np.concatenate([_sparse(rng, pre, D), batch, _sparse(rng, post, D)])
    d = np.arange(D)
    x[pre + B + d % post, d] = np.maximum(x[pre + B + d % post, d], 1.0)
    return x


def _empty_rows(rng):
    b = _sparse(rng, 200, 300)
    b[0] = 0
    b[-1] = 0
    b[60:68] = 0
    return Case("empty_rows", _frame(rng, b, 37), 37, 200)


def _empty_cols(rng):
    b = rng.poisson(0.6, size=(200, 300)).astype(np.float32)
    b[:, 0] = 0
    b[:, -1] = 0
    b[:, 100:110] = 0          # every column of this case is hot: these are hot columns empty in the batch
    return Case("empty_cols", _frame(rng, b, 21), 21, 200)


def _row_lengths(rng):
    """Rows of 0..9 cold entries (2U+1 for U = 4) after 0..2 hot ones: over a period of 30 rows every length
    0..9 occurs, and the period adds 165 = 1 (mod 4) entries, so 4 periods meet every row-pointer residue."""
    D = 300
    rows = []
    for r in range(120):
        L, h = r % 10, r % 3
        row = np.zeros(D, np.float32)
        row[rng.choice(64, h, replace=False)] = rng.integers(1, 6, size=h)
        row[128 + rng.choice(D - 128, L, replace=False)] = rng.integers(1, 6, size=L)
        rows.append(row)
    b = np.stack(rows)
    pre = _sparse(rng, 40, D, p_cold=0.0)
    x = np.concatenate([pre, b, np.zeros((4, D), np.float32)])
    d = np.arange(D)
    x[160 + d % 4, d] = np.maximum(x[160 + d % 4, d], 1.0)
    return x


def _long_column(rng):
    """B = 1600 rows.  In the batch's CSC the first columns hold 256, 0, 100, 156, 1600 (the whole column),
    192 and 1 entries: column starts at 256, 256, 512 and 2304 lie on 256-entry slice boundaries, the full column
    covers slices 2..7 entirely and straddles into slice 8."""
    B, D = 1600, 300
    b = _sparse(rng, B, D, p_hot=0.0, p_cold=0.01)
    b[:, 200:280] = np.where(rng.random((B, 80)) < 0.2, rng.integers(1, 6, size=(B, 80)), 0)
    b[:, :7] = 0
    for d, n in enumerate((256, 0, 100, 156, B, 192, 1)):
        b[rng.choice(B, n, replace=False), d] = rng.integers(1, 9, size=n)
    b[:, 7:96] = np.where(rng.random((B, 89)) < 0.06, 1.0, 0.0)
    return Case("long_column", _frame(rng, b, 9), 9, B)


def _long_rows(rng):
    """D = 4096: three full rows (4096 entries, longer than the hot split's 2048-entry stash) with counts 1..300."""
    B, D = 96, 4096
    b = _sparse(rng, B, D, hot=128, p_hot=0.3, p_cold=0.005)
    for r in (3, 40, 95):
        b[r] = rng.integers(1, 301, size=D)
    return Case("long_rows", _frame(rng, b, 11), 11, B)


LARGE_COUNTS = (63.0, 64.0, 65.0, 254.0, 255.0, 256.0, 70000.0,     # lgamma table edge, u8 overflow, > uint16
                2.5, 0.75, 96.5,                                     # non-integers bf16 holds exactly
                1.1, 300.7, 257.0)                                   # ... and ones it does not


def _large_counts(rng):
    b = _sparse(rng, 150, 300)
    for i, v in enumerate(LARGE_COUNTS):
        rows = rng.choice(150, 6, replace=False)
        b[rows, (7 * i) % 300] = v                  # hot columns
        b[rows, 150 + 9 * i] = v                    # cold columns
    b[17, :] = 0
    b[17, 5] = 70000.0                              # a row holding only one huge count
    return Case("large_counts", _frame(rng, b, 5), 5, 150)


def _rows(rng, B):
    b = rng.poisson(0.8, size=(B, 160)).astype(np.float32)
    b[:, 130:] = np.where(rng.random((B, 30)) < 0.02, 1.0, 0.0)     # a few cold columns
    return Case(f"rows_{B}", _frame(rng, b, 13, post=40), 13, B)


def make_case(name):
    rng = np.random.default_rng(sum(map(ord, name.split('@')[0])))
    if name == "empty_rows":
        return _empty_rows(rng)
    if name == "empty_cols":
        return _empty_cols(rng)
    if name.startswith("row_lengths@"):            # the same rows, cut at two offsets
        start = int(name.split("@")[1])
        return Case(name, _row_lengths(rng), 40 + start, 120 - start)
    if name == "long_column":
        return _long_column(rng)
    if name == "long_rows":
        return _long_rows(rng)
    if name == "large_counts":
        return _large_counts(rng)
    if name.startswith("rows_"):
        return _rows(rng, int(name.split("_")[1]))
    raise ValueError(name)


POISSON_CASES = ["empty_rows", "empty_cols", "row_lengths@0", "row_lengths@3", "long_column", "long_rows",
                 "large_counts", "rows_1", "rows_129", "rows_300"]
DENSE_LINK_CASES = ["empty_rows", "empty_cols", "row_lengths@0", "large_counts", "rows_650"]


# ------------------------------------------------------------------ metrics
def worst_ratio(got, ref, M):
    """max |got - ref| / M over the elements (the element-wise check is this <= rtol)."""
    got = np.asarray(got, dtype=np.float64)
    return float((np.abs(got - ref) / np.maximum(M, 1e-300)).max())


# feature axis of every Normal-family gradient tensor: v (K,D), w (1,D), u (D,K), s (2,D)
FEATURE_AXIS = {'v': 1, 'w': 1, 'u': 0, 's': 1}


def per_slice_rel_err(got, ref, axis, floor=1e-7):
    """Largest error of each slice along `axis` (a feature, or a row) over the largest |ref| of that slice,
    floored at `floor` times the largest |ref| of the whole tensor; the worst slice is returned."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    other = tuple(i for i in range(ref.ndim) if i != axis % ref.ndim)
    err = np.abs(got - ref).max(axis=other) if other else np.abs(got - ref)
    scale = np.abs(ref).max(axis=other) if other else np.abs(ref)
    return float((err / np.maximum(scale, floor * np.abs(ref).max() + 1e-300)).max())
