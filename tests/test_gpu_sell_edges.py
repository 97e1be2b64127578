"""GPU: the tiled SELL-32 Jacobian operator at the edges of its layout, row by row against an extended-precision product.

Every product with the Jacobian (jprod / jtprod, every Krylov step, the persistent loop) reads the layout `upload_sell`
builds: rows longer than 96 entries in a CSR of their own, 1 to 8 slices per tile with odd, even or zero widths, tiles
that mix slices with long rows or hold none, u16 windows, multi-segment windows or global int32 indices, odd windows at
the vector's end, row cuts into a multiple of the grid.  Each structure below is built by a named generator from a fixed
seed to reach one of those branches, and asserts through `B200Handle.tile_layout()` that the builder took it.

The bar is componentwise: for y = A x from raw COO entries (duplicates summed as given), every row i must satisfy
|y_i - y_ref_i| <= (L_i + 10) 2^-53 sum_k |a_k x_k|, with L_i the row's raw entry count and y_ref computed in long double;
empty rows must be exactly 0.  The bound covers a SELL row's two interleaved FMA chains and their final add, and a long
row's per-thread chains of about L / 256 terms followed by an 8-level tree.  Rows are scaled by 10^U(-12, 12) (columns
for the A' products), so an error confined to a row of small magnitude, which a norm-wise check cannot see, fails here
and the message names the row.

Run-time switches (`FPSB_LOOP=0`, `FPSB_NO_SEGS=1`) are read once per process, so the Krylov recurrences and the
single-window fallback of the multi-segment structures run in worker processes:
`python tests/test_gpu_sell_edges.py --worker <loop|step|noseg> <num_sms> <out.npz>`.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

LD = np.longdouble
if np.finfo(LD).nmant < 63:
    pytest.skip(f"np.longdouble has {np.finfo(LD).nmant} mantissa bits here; the reference needs at least 63",
                allow_module_level=True)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = LD(2.0) ** -53
LONG_ROW = 96           # kLongRow of fpsb_krylov.cu
WIN_CAP = 1536          # kWinCapMax
SEG_CAP = 1664          # kSegCapMax
MIN_GAP = 32            # kMinGap
KRYLOV_KS = (3, 8)
LAYOUT_KEYS = ("tiles", "windowed", "multi_segment", "global", "odd_window", "long_rows", "no_slices", "mixed")


# ---------------------------------------------------------------------------------------------------------------------
# structures: rows, cols (0-based COO, in the order handed to fpsb_create), base values, and the layout each one is for
# ---------------------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, m, n, rows, cols, base=None, index_base=0, seed=0, expect=None, segments=None):
        self.m, self.n = int(m), int(n)
        self.rows = np.asarray(rows, dtype=np.int64)
        self.cols = np.asarray(cols, dtype=np.int64)
        rng = np.random.default_rng(seed + 7)
        if base is None:
            base = rng.uniform(0.5, 2.0, self.rows.size) * rng.choice([-1.0, 1.0], self.rows.size)
        self.base = np.asarray(base, dtype=np.float64)
        self.index_base = index_base
        self.seed = seed
        self.expect = expect or {}
        self.segments = segments          # the window segments (start, length) of tile 0 of A, when multi-segment

    def matrix(self, vals=None):
        v = self.base if vals is None else vals
        return sp.csr_matrix((v, (self.rows, self.cols)), shape=(self.m, self.n))     # sums duplicates

    def row_len(self):
        return np.bincount(self.rows, minlength=self.m)

    def col_len(self):
        return np.bincount(self.cols, minlength=self.n)


def _rows_to_coo(col_lists):
    rows = np.concatenate([np.full(len(c), i, dtype=np.int64) for i, c in enumerate(col_lists)] + [np.zeros(0, np.int64)])
    cols = np.concatenate([np.asarray(c, dtype=np.int64) for c in col_lists] + [np.zeros(0, np.int64)])
    return rows, cols


def _spread(cols, m, rng):
    """Deal the given distinct columns out to m rows (round robin after a shuffle)."""
    cols = rng.permutation(np.asarray(cols, dtype=np.int64))
    return [cols[i::m] for i in range(m)]


def gen_long_cut(G):
    """Rows of 95, 96, 97 and 98 entries interleaved with short rows; dense columns of 96 and 97 entries."""
    rng = np.random.default_rng(101)
    m, n = 512, 3000
    pool = np.arange(2, n)
    cl = []
    for i in range(m):
        L = {0: 95, 1: 96, 2: 97, 3: 98}.get(i % 8, int(rng.integers(1, 8)))
        cl.append(list(rng.choice(pool, L, replace=False)))
    short = [i for i in range(m) if i % 8 >= 4]
    for c, k in ((0, 96), (1, 97)):
        for r in rng.choice(short, k, replace=False):
            cl[r].append(c)
    rows, cols = _rows_to_coo(cl)
    rl = np.bincount(rows, minlength=m)
    assert set(rl[np.arange(m) % 8 < 4]) == {95, 96, 97, 98} and rl[np.arange(m) % 8 >= 4].max() <= 9
    assert np.bincount(cols, minlength=n)[:2].tolist() == [96, 97]
    return Case(m, n, rows, cols, seed=101, expect=dict(A=dict(mixed=">0"), At=dict(long_rows=1, mixed=">0")))


def gen_all_long(G):
    """Every row longer than the SELL limit: every tile of A has no slice (ns = 0)."""
    rng = np.random.default_rng(102)
    m, n = 40, 3000
    cl = [rng.choice(n, int(rng.integers(97, 400)), replace=False) for _ in range(m)]
    rows, cols = _rows_to_coo(cl)
    return Case(m, n, rows, cols, seed=102, expect=dict(A=dict(long_rows=m, no_slices="tiles", mixed="tiles")))


SLICE_ROWS = (1, 31, 32, 33, 63, 64, 255, 256, 257)


def _slices(nrows):
    """Row lengths 0..9 (odd, even, zero slice widths); in the first tile at least the last slice's worth of rows is
    empty, so its last slice is all padding (width 0); with 257 rows the second tile has no entries at all."""
    rng = np.random.default_rng(200 + nrows)
    n = 600
    lens = rng.integers(1, 10, nrows)
    if nrows == 1:
        lens[:] = 3
    for t0 in range(0, min(nrows, 256), 256):
        k = min(nrows, 256) - t0
        last = k - 32 * ((k - 1) // 32)
        if k > 32:
            lens[t0 + rng.choice(k, max(last, k // 3), replace=False)] = 0
    lens[256:] = 0
    cl = [rng.choice(n, int(L), replace=False) for L in lens]
    rows, cols = _rows_to_coo(cl)
    # the slice widths of the first tile: odd, even and zero ones (rows sorted by length, 32 to a slice)
    w = [int(x) for x in np.sort(lens[:256])[::-1][::32]]
    if nrows > 32:
        assert w[-1] == 0, w
    if nrows >= 255:
        assert any(x % 2 for x in w) and any(x % 2 == 0 and x > 0 for x in w), w
    ntiles = (nrows + 255) // 256
    exp = dict(tiles=ntiles, windowed=1, **{"global": ntiles - 1})
    return Case(nrows, n, rows, cols, seed=200 + nrows, expect=dict(A=exp))


def _strided(m, n, ncols, extra=()):
    """m rows, row r holding columns r, r + m, r + 2m, ... below ncols, plus `extra` (row, col) entries."""
    cl = [list(range(r, ncols, m)) for r in range(m)]
    for r, c in extra:
        cl[r].append(c)
    return _rows_to_coo(cl)


def gen_win_exact(G):
    """One tile whose column span is exactly the 1536-entry window capacity."""
    rows, cols = _strided(32, 1600, WIN_CAP)
    return Case(32, 1600, rows, cols, seed=103, expect=dict(A=dict(tiles=1, windowed=1, multi_segment=0, odd_window=0)))


def gen_win_1537(G):
    """A span of 1537: one past the capacity, no gap to cut at: global indices."""
    rows, cols = _strided(32, 1600, WIN_CAP, extra=[(0, WIN_CAP)])
    return Case(32, 1600, rows, cols, seed=104, expect=dict(A=dict(tiles=1, windowed=0, **{"global": 1})))


def gen_win_dropped(G):
    """32 rows of 96 entries over a span of 1000: the window fits the capacity but not the stage next to the slice, and
    a single slice cannot be split: the window is dropped."""
    rng = np.random.default_rng(105)
    cl = [rng.choice(1000, LONG_ROW, replace=False) for _ in range(32)]
    rows, cols = _rows_to_coo(cl)
    return Case(32, 1200, rows, cols, seed=105, expect=dict(A=dict(tiles=1, windowed=0, long_rows=0, **{"global": 1})))


def gen_win_odd_end(G):
    """A window that ends at the last column of an odd ncols: odd length (window copied by the consumer groups)."""
    rng = np.random.default_rng(106)
    m, n = 64, 701
    cl = [rng.choice(np.arange(600, n), int(rng.integers(1, 8)), replace=False) for _ in range(m)]
    cl[0] = np.r_[600, 700]
    rows, cols = _rows_to_coo(cl)
    return Case(m, n, rows, cols, seed=106, expect=dict(A=dict(tiles=1, windowed=1, odd_window=1)))


def _runs(name_seed, runs, n, m=32, step=8):
    """Columns of a few runs [start, start + len) (every `step`-th column and both ends), dealt out to m rows."""
    rng = np.random.default_rng(name_seed)
    cs = set()
    for s, L in runs:
        cs.update(range(s, s + L, step))
        cs.add(s + L - 1)
    u = np.array(sorted(cs))
    return _rows_to_coo(_spread(u, m, rng)), u


def _gaps_case(g, seed, segments):
    """Three runs far apart, the middle one split by a gap of g columns: cut from kMinGap = 32 on."""
    runs = [(0, 200), (1200, 100), (1299 + g, 100), (3000, 200)]
    (rows, cols), u = _runs(seed, runs, 3300)
    d = np.diff(u)
    assert g in d.tolist() and (d >= MIN_GAP).sum() == 2 + (g >= MIN_GAP) and u[-1] - u[0] + 1 > WIN_CAP
    return Case(32, 3300, rows, cols, seed=seed, expect=dict(A=dict(tiles=1, windowed=1, multi_segment=1)),
                segments=segments)


def gen_gap31(G):
    """A gap of 31 stays inside the segment [1200, 1430)."""
    return _gaps_case(31, 111, [(0, 200), (1200, 230), (3000, 200)])


def gen_gap32(G):
    """A gap of 32 is cut; the run after it starts at an odd column (1331): its segment starts one earlier and is
    rounded up to an even length."""
    return _gaps_case(32, 112, [(0, 200), (1200, 100), (1330, 102), (3000, 200)])


def gen_gap33(G):
    return _gaps_case(33, 113, [(0, 200), (1200, 100), (1332, 100), (3000, 200)])


def gen_gaps_equal(G):
    """Five runs with four equal qualifying gaps: only three are cut, the leftmost ones."""
    runs = [(600 * k, 100) for k in range(5)]
    (rows, cols), u = _runs(114, runs, 2600)
    d = np.diff(u)
    assert (d >= MIN_GAP).sum() == 4 and len(set(d[d >= MIN_GAP].tolist())) == 1
    return Case(32, 2600, rows, cols, seed=114, expect=dict(A=dict(tiles=1, windowed=1, multi_segment=1)),
                segments=[(0, 100), (600, 100), (1200, 100), (1800, 700)])


def _segcap_case(last, seed):
    runs = [(0, 554), (1554, 554), (3108, last)]
    (rows, cols), u = _runs(seed, runs, 3108 + last + 10)
    return Case(32, 3108 + last + 10, rows, cols, seed=seed), 554 + 554 + last


def gen_segcap_under(G):
    """Three segments of 1664 entries in all: exactly kSegCapMax."""
    c, tot = _segcap_case(556, 115)
    assert tot == SEG_CAP
    c.expect = dict(A=dict(tiles=1, windowed=1, multi_segment=1))
    c.segments = [(0, 554), (1554, 554), (3108, 556)]
    return c


def gen_segcap_over(G):
    """Three segments of 1666 entries: over kSegCapMax, global indices."""
    c, tot = _segcap_case(558, 116)
    assert tot == SEG_CAP + 2
    c.expect = dict(A=dict(tiles=1, windowed=0, multi_segment=0, **{"global": 1}))
    return c


def gen_coo(G):
    """Unsorted COO with the same (i, j) repeated at distant positions, explicit zeros, one-based indices."""
    rng = np.random.default_rng(117)
    m, n = 300, 500
    cl = [np.clip(i * n // m + rng.choice(np.arange(-20, 20), 6, replace=False), 0, n - 1) for i in range(m)]
    cl = [np.unique(c) for c in cl]
    rows, cols = _rows_to_coo(cl)
    p = rng.permutation(rows.size)
    rows, cols = rows[p], cols[p]
    dup = rng.choice(rows.size, rows.size // 8, replace=False)
    dup = dup[np.argsort(-dup)]                     # repeats of late entries early in the tail and vice versa
    rows, cols = np.r_[rows, rows[dup]], np.r_[cols, cols[dup]]
    c = Case(m, n, rows, cols, index_base=1, seed=117,
             expect=dict(A=dict(tiles=2, windowed=2, long_rows=0), At=dict(tiles=2, windowed=2, long_rows=0)))
    c.base[rng.choice(rows.size, rows.size // 20, replace=False)] = 0.0
    assert len(set(zip(rows.tolist(), cols.tolist()))) < rows.size
    return c


def gen_m1(G):
    rng = np.random.default_rng(118)
    rows, cols = _rows_to_coo([rng.choice(300, 60, replace=False)])
    return Case(1, 300, rows, cols, seed=118, expect=dict(A=dict(tiles=1)))


def gen_n1(G):
    """One column: A' is a single row of 210 entries (long, no slice)."""
    rng = np.random.default_rng(119)
    m = 300
    cl = [[0] if k else [] for k in rng.random(m) < 0.7]
    rows, cols = _rows_to_coo(cl)
    return Case(m, 1, rows, cols, seed=119, expect=dict(At=dict(tiles=1, long_rows=1, no_slices=1)))


def gen_tall(G):
    rng = np.random.default_rng(120)
    m, n = 500, 120
    rows, cols = _rows_to_coo([rng.choice(n, 4, replace=False) for _ in range(m)])
    return Case(m, n, rows, cols, seed=120, expect=dict(A=dict(tiles=2, windowed=2), At=dict(tiles=1, windowed=1)))


def gen_empty_edges(G):
    """Empty first and last rows and columns."""
    rng = np.random.default_rng(121)
    m, n = 300, 400
    cl = [[] if i in (0, m - 1) else rng.choice(np.arange(1, n - 1), 5, replace=False) for i in range(m)]
    rows, cols = _rows_to_coo(cl)
    assert 0 not in cols and n - 1 not in cols
    return Case(m, n, rows, cols, seed=121, expect=dict(A=dict(tiles=2, windowed=2), At=dict(tiles=2, windowed=2)))


def _band(m, n, seed):
    rng = np.random.default_rng(seed)
    base = (np.arange(m) * (n - 3)) // max(m - 1, 1)
    cols = (base[:, None] + np.array([0, 1, 2])[None, :]).ravel()
    rows = np.repeat(np.arange(m), 3)
    keep = rng.random(rows.size) < 0.9
    return rows[keep], cols[keep]


def gen_rowcut_below(G):
    """4 x num_sms - 1 tiles of 256 rows: no row cuts."""
    m = 256 * (4 * G - 1)
    rows, cols = _band(m, m // 2, 122)
    return Case(m, m // 2, rows, cols, seed=122, expect=dict(A=dict(tiles=4 * G - 1)))


def gen_rowcut_above(G):
    """One row past 4 x num_sms tiles: the rows are re-cut into a multiple of the grid (5 x num_sms tiles)."""
    m = 256 * 4 * G + 1
    rows, cols = _band(m, m // 2, 123)
    return Case(m, m // 2, rows, cols, seed=123, expect=dict(A=dict(tiles=5 * G)))


GENERATORS = {
    "long_cut": gen_long_cut, "all_long": gen_all_long,
    **{f"slices{r}": (lambda G, r=r: _slices(r)) for r in SLICE_ROWS},
    "win_exact": gen_win_exact, "win_1537": gen_win_1537, "win_dropped": gen_win_dropped, "win_odd_end": gen_win_odd_end,
    "gap31": gen_gap31, "gap32": gen_gap32, "gap33": gen_gap33, "gaps_equal": gen_gaps_equal,
    "segcap_under": gen_segcap_under, "segcap_over": gen_segcap_over,
    "coo": gen_coo, "m1": gen_m1, "n1": gen_n1, "tall": gen_tall, "empty_edges": gen_empty_edges,
    "rowcut_below": gen_rowcut_below, "rowcut_above": gen_rowcut_above,
}
NAMES = list(GENERATORS)
MULTISEG = ["gap31", "gap32", "gap33", "gaps_equal", "segcap_under"]
ROWCUT = ["rowcut_below", "rowcut_above"]
_CASES = {}


def case(name, G):
    if (name, G) not in _CASES:
        _CASES[(name, G)] = GENERATORS[name](G)
    return _CASES[(name, G)]


def check_layout(c, lay, H):
    """The branch the generator is for, plus what must hold for every operator."""
    if c.segments is not None:
        assert H.tile_segments(0) == c.segments, H.tile_segments(0)
    for op, L, lens in (("A", lay["A"], c.row_len()), ("At", lay["At"], c.col_len())):
        assert L["long_rows"] == int((lens > LONG_ROW).sum()), (op, L)
        assert L["windowed"] + L["global"] == L["tiles"] and L["multi_segment"] <= L["windowed"], (op, L)
        assert L["odd_window"] <= L["windowed"] and L["no_slices"] <= L["mixed"] <= L["tiles"], (op, L)
        if L["long_rows"] == 0:
            assert L["mixed"] == 0, (op, L)
        for k, want in c.expect.get(op, {}).items():
            got = L[k]
            if want == ">0":
                assert got > 0, (op, k, L)
            elif want == "tiles":
                assert got == L["tiles"] and got > 0, (op, k, L)
            else:
                assert got == want, (op, k, L)


# ---------------------------------------------------------------------------------------------------------------------
# the reference and the bar
# ---------------------------------------------------------------------------------------------------------------------
def _distinct(rng, n, k):
    """k columns of n distinct magnitudes in [1, 2], random signs."""
    base = np.linspace(1.0, 2.0, max(n, 1))[:n]
    return np.stack([rng.permutation(base) * rng.choice([-1.0, 1.0], n) for _ in range(k)], axis=1)


def reference(rows, cols, vals, X, nout):
    """y = A X over the raw entries in long double, s = sum |a x| and the raw entry count of every output row."""
    X = np.asarray(X, dtype=np.float64).reshape(X.shape[0], -1)
    prod = vals.astype(LD)[:, None] * X[cols].astype(LD)
    y = np.zeros((nout, X.shape[1]), dtype=LD)
    s = np.zeros((nout, X.shape[1]), dtype=LD)
    np.add.at(y, rows, prod)
    np.add.at(s, rows, np.abs(prod))
    return y, s, np.bincount(rows, minlength=nout)


def bar_ratio(got, ref, col, what):
    """Componentwise check of one output column; returns the worst error / bound ratio."""
    y, s, L = ref[0][:, col], ref[1][:, col], ref[2]
    got = np.asarray(got, dtype=np.float64)
    err = np.abs(got.astype(LD) - y)
    bound = (L.astype(LD) + 10) * U * s
    bad = err > bound
    bad |= (L == 0) & (got != 0.0)
    bad |= ~np.isfinite(got)
    if bad.any():
        ratio = np.where(bound > 0, err / np.where(bound > 0, bound, 1), np.inf)
        worst = np.argsort(-np.where(bad, ratio, -1))[:5]
        lines = [f"row {i}: {L[i]} entries, bound {float(bound[i]):.3e}, error {float(err[i]):.3e}, "
                 f"got {got[i]!r}, want {float(y[i])!r}" for i in worst if bad[i]]
        raise AssertionError(f"{what}: {int(bad.sum())} of {got.size} rows off the componentwise bar\n  " + "\n  ".join(lines))
    with np.errstate(invalid="ignore", divide="ignore"):
        r = np.where(bound > 0, err / np.where(bound > 0, bound, 1), 0)
    return float(r.max()) if r.size else 0.0


def value_sets(c):
    """Row-scaled values (the A products see errors in small rows), column-scaled ones (the A' products), and a second
    row-scaled set; explicit zeros stay zero."""
    rng = np.random.default_rng(c.seed + 1)
    rs1 = 10.0 ** rng.uniform(-12, 12, c.m)
    cs2 = 10.0 ** rng.uniform(-12, 12, c.n)
    rs3 = 10.0 ** rng.uniform(-12, 12, c.m)
    return [c.base * rs1[c.rows], c.base * cs2[c.cols], c.base * rs3[c.rows]]


# ---------------------------------------------------------------------------------------------------------------------
# helpers on the GPU side
# ---------------------------------------------------------------------------------------------------------------------
def make_handle(c):
    import fpsb200
    return fpsb200.B200Handle(c.n, c.m, c.rows + c.index_base, c.cols + c.index_base, index_base=c.index_base)


def _fixed_opts(n, m, k):
    import ctypes
    import fpsb200
    o = fpsb200.IterOpts()
    fpsb200._lib.lib().fpsb_iter_default_opts(ctypes.c_int64(n), ctypes.c_int64(m), ctypes.byref(o))
    for name, v in dict(ls_atol=0.0, ls_rtol=0.0, ls_itmax=k, ln_atol=0.0, ln_rtol=0.0, ln_btol=0.0, ln_itmax=k,
                        ne_atol=0.0, ne_rtol=0.0, ne_etol=0.0, ne_itmax=k).items():
        setattr(o, name, v)
    return o


def _np(a):
    return a if isinstance(a, np.ndarray) else a.cpu().numpy()


ENTRIES = ("host", "pinned", "device", "offset")


def _call(H, fn, x, entry):
    """One product with the input in host memory, page-locked host memory, a device tensor, or a device tensor one
    element into its buffer (8- but not 16-byte aligned: the windows are staged by the consumer groups)."""
    import torch
    x = np.ascontiguousarray(x)
    if entry == "host":
        return fn(x)
    if entry == "pinned":
        H.pin_host(x)
        try:
            return fn(x)
        finally:
            H.unpin_host(x)
    t = torch.zeros(x.size + 1, dtype=torch.float64, device="cuda")
    if entry == "device":
        t = t[:x.size]
        t.copy_(torch.as_tensor(x))
    else:
        t[1:] = torch.as_tensor(x)
        t = t[1:]
        assert t.data_ptr() % 16 == 8
    return _np(fn(t))


def check_products(H, c, vals, rng, what):
    """jprod, jprod2, jtprod, jtprod2 through every entry, each on fresh inputs; returns the worst ratio."""
    X = _distinct(rng, c.n, 3 * len(ENTRIES))
    Uv = _distinct(rng, c.m, 3 * len(ENTRIES))
    ra = reference(c.rows, c.cols, vals, X, c.m)
    rt = reference(c.cols, c.rows, vals, Uv, c.n)
    worst = 0.0
    for e, entry in enumerate(ENTRIES):
        j = 3 * e
        worst = max(worst, bar_ratio(_call(H, H.jprod, X[:, j], entry), ra, j, f"{what} jprod {entry}"))
        y2 = _call(H, H.jprod2, np.r_[X[:, j + 1], X[:, j + 2]], entry)
        worst = max(worst, bar_ratio(y2[:c.m], ra, j + 1, f"{what} jprod2[0] {entry}"),
                    bar_ratio(y2[c.m:], ra, j + 2, f"{what} jprod2[1] {entry}"))
        worst = max(worst, bar_ratio(_call(H, H.jtprod, Uv[:, j], entry), rt, j, f"{what} jtprod {entry}"))
        z2 = _call(H, H.jtprod2, np.r_[Uv[:, j + 1], Uv[:, j + 2]], entry)
        worst = max(worst, bar_ratio(z2[:c.n], rt, j + 1, f"{what} jtprod2[0] {entry}"),
                    bar_ratio(z2[c.n:], rt, j + 2, f"{what} jtprod2[1] {entry}"))
    return worst


@pytest.fixture(scope="session")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# 1-3. layout, products through every entry, value refresh, batched CSR products
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", NAMES)
def test_layout_and_products(name, num_sms):
    """The layout the structure is for; every product through every entry after a refresh from host memory, from a
    device tensor, and from host memory again after a Krylov solve on the same handle."""
    import torch
    c = case(name, num_sms)
    H = make_handle(c)
    lay = H.tile_layout()
    check_layout(c, lay, H)
    st = H.tile_stats()
    for op in ("A", "At"):
        assert [st[op][k] for k in ("tiles", "windowed", "multi_segment")] == \
               [lay[op][k] for k in ("tiles", "windowed", "multi_segment")]
    rng = np.random.default_rng(c.seed + 2)
    v1, v2, v3 = value_sets(c)
    worst = {}
    H.set_jac_values(v1)
    worst["host values"] = check_products(H, c, v1, rng, f"{name} (host values)")
    H.set_jac_values(torch.as_tensor(v2, device="cuda"))
    worst["device values"] = check_products(H, c, v2, rng, f"{name} (device values)")
    H.iter_setup(_fixed_opts(c.n, c.m, 5))
    H.iter_solve_two_mixed(1e-2, rng.standard_normal(c.n), rng.standard_normal(c.m))
    H.set_jac_values(v3)
    worst["after a solve"] = check_products(H, c, v3, rng, f"{name} (after a Krylov solve)")
    print(f"\n{name}: A {lay['A']}  A' {lay['At']}  worst error / bound " +
          " ".join(f"{k}: {v:.3f}" for k, v in worst.items()))


@pytest.mark.parametrize("name", [n for n in NAMES if n not in ROWCUT])
def test_batched_csr_products(name, num_sms):
    """batch_jprod / batch_jtprod (plain CSR kernels) with one set of values and with one set per instance."""
    import torch
    c = case(name, num_sms)
    H = make_handle(c)
    vs = value_sets(c)
    rng = np.random.default_rng(c.seed + 3)
    X = _distinct(rng, c.n, 3)
    Uv = _distinct(rng, c.m, 3)
    Xt, Ut = torch.as_tensor(X.T.copy(), device="cuda"), torch.as_tensor(Uv.T.copy(), device="cuda")
    shared = _np(H.batch_jprod(torch.as_tensor(vs[0], device="cuda"), Xt))
    sharedt = _np(H.batch_jtprod(torch.as_tensor(vs[1], device="cuda"), Ut))
    per = _np(H.batch_jprod(torch.as_tensor(np.stack(vs), device="cuda"), Xt))
    pert = _np(H.batch_jtprod(torch.as_tensor(np.stack(vs), device="cuda"), Ut))
    ra = reference(c.rows, c.cols, vs[0], X, c.m)
    rt = reference(c.cols, c.rows, vs[1], Uv, c.n)
    for i in range(3):
        bar_ratio(shared[i], ra, i, f"{name} batch_jprod shared values, instance {i}")
        bar_ratio(sharedt[i], rt, i, f"{name} batch_jtprod shared values, instance {i}")
        bar_ratio(per[i], reference(c.rows, c.cols, vs[i], X[:, i:i + 1], c.m), 0, f"{name} batch_jprod instance {i}")
        bar_ratio(pert[i], reference(c.cols, c.rows, vs[i], Uv[:, i:i + 1], c.n), 0, f"{name} batch_jtprod instance {i}")


DIST_NAMES = [n for n in NAMES if n not in ROWCUT]


@pytest.mark.parametrize("name", DIST_NAMES)
def test_partitioned_handle_world1(name, num_sms):
    """The row-partitioned handle at world size 1 builds its own tiles from the same builder."""
    from fpsb200.partition import DistHandle, RowPartition
    c = case(name, num_sms)
    D = DistHandle(RowPartition(c.n, c.m, c.rows, c.cols, 1), 0, device=0)
    rng = np.random.default_rng(c.seed + 4)
    for k, v in enumerate(value_sets(c)[:2]):
        D.set_jac_values(v)
        X = _distinct(rng, c.n, 1)
        Uv = _distinct(rng, c.m, 1)
        bar_ratio(D.jprod(X[:, 0]), reference(c.rows, c.cols, v, X, c.m), 0, f"{name} dist jprod, values {k}")
        bar_ratio(D.jtprod(Uv[:, 0]), reference(c.cols, c.rows, v, Uv, c.n), 0, f"{name} dist jtprod, values {k}")


def test_tile_layout_of_empty_operator():
    import fpsb200
    H = fpsb200.B200Handle(7, 0, np.zeros(0, np.int64), np.zeros(0, np.int64))
    lay = H.tile_layout()
    assert all(v == 0 for v in lay["A"].values()), lay
    assert lay["At"]["long_rows"] == 0 and lay["At"]["mixed"] == 0, lay
    assert H.tile_segments(0, transpose=True) == []
    with pytest.raises(fpsb200.FpsbError, match="out of range"):
        H.tile_segments(0)


# ---------------------------------------------------------------------------------------------------------------------
# 4. Krylov recurrences on the same layouts (persistent loop and step path, in worker processes)
# ---------------------------------------------------------------------------------------------------------------------
# rank 1 operators exhaust their Krylov space in one iteration: past it the recurrences run on roundoff
KRYLOV_NAMES = [n for n in NAMES if n not in ("m1", "n1", "slices1")]
KINDS = (("mixed0", "mixed", 0.0), ("mixed2", "mixed", 1e-2), ("ls", "ls", 1e-2), ("extras", "extras", 1e-2))
LOOP_KEYS = ("persistent", "early", "nstage", "grid", "stage_bytes", "inflight", "nspec", "chunk")


def _krylov_rhs(c):
    rng = np.random.default_rng(c.seed + 5)
    return rng.standard_normal(c.n), rng.standard_normal(c.m), rng.standard_normal(c.n)


def _work_krylov(out, G):
    for name in KRYLOV_NAMES:
        c = case(name, G)
        H = make_handle(c)
        H.set_jac_values(c.base)
        out[f"{name}.layout"] = np.array([H.tile_layout()[op][k] for op in ("A", "At") for k in LAYOUT_KEYS])
        r1, r2, r3 = _krylov_rhs(c)
        for k in KRYLOV_KS:
            H.iter_setup(_fixed_opts(c.n, c.m, k))
            for key, kind, d in KINDS:
                if kind == "mixed":
                    got = H.iter_solve_two_mixed(d, r1, r2)
                elif kind == "ls":
                    got = H.iter_solve_two_least_squares(d, r1, r3)
                else:
                    got = H.iter_solve_two_extras(d, r1, r2)
                tag = f"{name}.k{k}.{key}"
                for i, v in enumerate(got[:-1]):
                    out[f"{tag}.{i}"] = np.asarray(v)
                out[f"{tag}.niter"] = np.array([s["niter"] for s in got[-1]])
                out[f"{tag}.loop"] = np.array([H.loop_info()[q] for q in LOOP_KEYS])


def _work_noseg(out, G):
    for name in MULTISEG:
        c = case(name, G)
        H = make_handle(c)
        out[f"{name}.layout"] = np.array([H.tile_layout()[op][k] for op in ("A", "At") for k in LAYOUT_KEYS])
        out[f"{name}.segments"] = np.array(H.tile_segments(0)).reshape(-1, 2)
        v = value_sets(c)
        rng = np.random.default_rng(c.seed + 6)
        for j, vals in enumerate(v[:2]):
            H.set_jac_values(vals)
            X = _distinct(rng, c.n, 3)
            Uv = _distinct(rng, c.m, 3)
            out[f"{name}.v{j}.X"], out[f"{name}.v{j}.U"] = X, Uv
            out[f"{name}.v{j}.y"] = H.jprod(X[:, 0])
            out[f"{name}.v{j}.y2"] = H.jprod2(np.r_[X[:, 1], X[:, 2]])
            out[f"{name}.v{j}.z"] = H.jtprod(Uv[:, 0])
            out[f"{name}.v{j}.z2"] = H.jtprod2(np.r_[Uv[:, 1], Uv[:, 2]])


WORKERS = {"loop": ({}, _work_krylov), "step": ({"FPSB_LOOP": "0"}, _work_krylov), "noseg": ({"FPSB_NO_SEGS": "1"}, _work_noseg)}
WORKER_TIMEOUT = 300


@pytest.fixture(scope="session")
def runs(tmp_path_factory, num_sms):
    cache = {}
    base = tmp_path_factory.mktemp("sell_edges")

    def get(env):
        if env not in cache:
            path = str(base / f"{env}.npz")
            child = {k: v for k, v in os.environ.items() if not k.startswith("FPSB_")}
            child.update(WORKERS[env][0])
            child["PYTHONPATH"] = os.pathsep.join([ROOT] + [p for p in sys.path if p])
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--worker", env, str(num_sms), path],
                               env=child, cwd=ROOT, capture_output=True, text=True, timeout=WORKER_TIMEOUT)
            if r.returncode != 0:
                raise AssertionError(f"worker {env} exited with {r.returncode}:\n{r.stderr[-4000:]}")
            with np.load(path) as z:
                cache[env] = {k: z[k] for k in z.files}
        return cache[env]

    return get


_ORACLE = {}


def _oracle_run(oracle, c, name, k, kind, d):
    key = (name, k, kind, d)
    if key not in _ORACLE:
        A = c.matrix()
        r1, r2, r3 = _krylov_rhs(c)
        o = oracle.IterativeOracle(A, **dict(ls_atol=0.0, ls_rtol=0.0, ls_itmax=k, ln_atol=0.0, ln_rtol=0.0, ln_btol=0.0,
                                             ln_itmax=k, ne_atol=0.0, ne_rtol=0.0, ne_etol=0.0, ne_itmax=k))
        if kind == "mixed":
            _ORACLE[key] = o.solve_two_mixed(d, r1, r2)
        elif kind == "ls":
            _ORACLE[key] = o.solve_two_least_squares(d, r1, r3)
        else:
            _ORACLE[key] = o.solve_two_extras(d, r1, r2)
    return _ORACLE[key]


def _rel(a, b):
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300))


@pytest.mark.parametrize("env", ["loop", "step"])
def test_krylov_on_layout_edges(runs, oracle, env, num_sms):
    """LSQR / CRAIG / MINRES at 3 and 8 iterations, all tolerances 0: the oracle's iteration counts and iterates within
    1e-11.  Operators with long rows (or an empty operator side) cannot run the persistent loop: they take the step
    path in both workers."""
    r = runs(env)
    worst = {}
    for name in KRYLOV_NAMES:
        c = case(name, num_sms)
        lay = r[f"{name}.layout"]
        can_loop = lay[LAYOUT_KEYS.index("long_rows")] == 0 and lay[8 + LAYOUT_KEYS.index("long_rows")] == 0 \
            and lay[0] > 0 and lay[8] > 0
        for k in KRYLOV_KS:
            for key, kind, d in KINDS:
                tag = f"{name}.k{k}.{key}"
                li = dict(zip(LOOP_KEYS, r[f"{tag}.loop"].tolist()))
                assert li["persistent"] == (1 if env == "loop" and can_loop else 0), (tag, li)
                ref = _oracle_run(oracle, c, name, k, kind, d)
                assert r[f"{tag}.niter"].tolist() == [s["niter"] for s in ref[-1]], (tag, r[f"{tag}.niter"])
                for i in range(len(ref) - 1):
                    e = _rel(r[f"{tag}.{i}"], ref[i])
                    worst[name] = max(worst.get(name, 0.0), e)
                    assert e < 1e-11, (tag, i, e)
    print(f"\n{env}: worst relative difference to the oracle", {k: f"{v:.1e}" for k, v in worst.items()})
    assert any(dict(zip(LOOP_KEYS, r[f"{n}.k3.mixed0.loop"].tolist()))["persistent"] for n in KRYLOV_NAMES) == (env == "loop")


def test_multisegment_structures_without_segments(runs, num_sms):
    """FPSB_NO_SEGS=1: the same operators without multi-segment windows, held to the same componentwise bar (not
    bitwise: the entry order inside a row follows the window's bank groups)."""
    r = runs("noseg")
    for name in MULTISEG:
        c = case(name, num_sms)
        lay = dict(zip(LAYOUT_KEYS, r[f"{name}.layout"][:8].tolist()))
        assert lay["multi_segment"] == 0 and lay["global"] == lay["tiles"], lay
        assert r[f"{name}.segments"].size == 0
        for j, vals in enumerate(value_sets(c)[:2]):
            X, Uv = r[f"{name}.v{j}.X"], r[f"{name}.v{j}.U"]
            ra = reference(c.rows, c.cols, vals, X, c.m)
            rt = reference(c.cols, c.rows, vals, Uv, c.n)
            bar_ratio(r[f"{name}.v{j}.y"], ra, 0, f"{name} no segments jprod")
            bar_ratio(r[f"{name}.v{j}.y2"][:c.m], ra, 1, f"{name} no segments jprod2[0]")
            bar_ratio(r[f"{name}.v{j}.y2"][c.m:], ra, 2, f"{name} no segments jprod2[1]")
            bar_ratio(r[f"{name}.v{j}.z"], rt, 0, f"{name} no segments jtprod")
            bar_ratio(r[f"{name}.v{j}.z2"][:c.n], rt, 1, f"{name} no segments jtprod2[0]")
            bar_ratio(r[f"{name}.v{j}.z2"][c.n:], rt, 2, f"{name} no segments jtprod2[1]")


def _worker(argv):
    env, G, path = argv
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    out = {}
    WORKERS[env][1](out, int(G))
    np.savez(path, **out)


if __name__ == "__main__":
    if len(sys.argv) == 5 and sys.argv[1] == "--worker":
        _worker(sys.argv[2:])
    else:
        sys.exit("usage: python tests/test_gpu_sell_edges.py --worker <loop|step|noseg> <num_sms> <out.npz>")
