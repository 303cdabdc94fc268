"""The two event voxelisers against float64 accumulations of the reference's own per-event expressions.

Contract (event_voxel.cu): the kernels compute every per-event, per-tap weight in fp32, one rounded operation at a time
and in the reference's order (oracle/torch_ref.py restates event_utils.py and dsec.py with the same torch operators), so
each weight equals the reference's bit for bit.  Only the order in which the weights reach a cell differs (atomics).

Reference.  ref_int and ref_trilinear evaluate the expressions of torch_ref.events_to_voxel and
torch_ref.events_to_voxel_trilinear vectorised in NumPy fp32 (NumPy >= 2 keeps a Python scalar weak, as torch does, so
every operation rounds to fp32 as there; the test_*_reference_matches_torch_ref tests check it), then accumulate the fp32 weights
into a float64 grid.  Per cell they also keep the number m of contributions that are not zero and their sum S = sum |w|.

Per-cell bar.  An fp32 sum of m terms in any order, starting from the zero fill, rounds m - 1 times; each rounding is at
most 2^-24 of a partial sum, and every partial sum is at most S, so |got - ref| <= (m - 1) 2^-24 S (1 + e).  The factor
1 + e = 1 + 2^-9 covers the second-order term of that bound, (m - 1) 2^-24 / (1 - (m - 1) 2^-24) - (m - 1) 2^-24, for
m < 2^14 (asserted), and the float64 rounding of ref and S (below 2^-53 m S).  So a cell with m = 1 must equal its one
weight exactly, a cell with m = 0 must be +0.0 bit for bit (the kernels add nothing to it, or only +-0), and NaN cells
of the reference must be NaN in the kernel's grid and nowhere else.

float64 event arrays (int voxeliser): the reference then computes its weights in float64 and rounds each to fp32,
while eventsToVoxel shifts the timestamps in float64 and casts them, so the kernel's fp32 chain
tn = ((t - t0) / den) / dt * (bins - 1) rounds six times more: |tn32 - tn64| <= 6 * 2^-24 |tn|, and the bin weight
1 - |tn - b| and the product with p round twice more on the kernel's side and once on the reference's.  Every event
whose |tn64 - b| < 1 + 1e-5 (it may contribute on either side) therefore adds |p| (6 bins + 3) 2^-24 to the bar and
counts in m.

Cases are named parameters.  Every small case runs with `out` at 0, 4, 8 and 12 bytes past a 16-byte boundary, inside a
buffer poisoned with a NaN payload: the floats around the slice must come back bit-unchanged and every float inside it
must be written.  The tri-linear kernel picks its store by address (a red.v2 when the left tap of an x pair is 8-byte
aligned; a red.v4 with zero outer lanes when it sits at 4 mod 16 and the four lanes stay inside the grid; scalar
atomics otherwise): test_store_paths_are_all_reached computes on the host the path each tap takes and checks that the
suite reaches all three, in both polarity planes, at all four alignments, and at the grid's first cell, its last pair,
row ends and the polarity plane boundary.

The bar is a rigorous bound, and it is tight: a two-term cell whose sum lands just above a power of two can reach it.
Largest measured |got - ref| / bar per case family on a B200 at its 1000 W power limit (the GPU tests of this file run
in about 35 s there, most of it the float64 references of the 4 M-event cases):
  int small 0.989, int things 0.998, int hd 0.998, int float64 0.254, int degenerate 0 (NaN cells and m <= 1 only),
  trilinear small 0.976, trilinear census 0.987, trilinear dsec 0.998, trilinear hd 0.998,
  batched dsec 0.998 (voxelise with 1 and 2 lanes), batched dsec graph 0.998, batched things 0.998.
"""
import functools
import itertools
import zlib

import numpy as np
import pytest
import torch

from oracle import torch_ref

U = 2.0 ** -24
POISON = 0x7FA00BAD                                     # a quiet NaN with a payload no kernel result carries
INT_MIN = -(2 ** 31)
MEASURED = {}                                           # family -> largest |got - ref| / bar seen


# ------------------------------------------------------------------------------------------------- reference
def _trunc_i32(v):
    """float -> int32 as x86 converts it (torch's .int(), NumPy's astype(int32)): toward zero; NaN, +-inf and values
    outside the int32 range become INT_MIN.  Returned as int64 so that +1 cannot overflow."""
    v = np.asarray(v)
    with np.errstate(invalid="ignore"):
        ok = np.abs(v) < 2.0 ** 31
    out = np.full(v.shape, INT_MIN, np.int64)
    out[ok] = np.trunc(v[ok]).astype(np.int64)
    return out


class _Grid:
    """float64 sum, contribution count m and sum |w| per cell (+ the widening term of float64 event arrays)."""

    def __init__(self, shape):
        self.shape = shape
        self.cells = int(np.prod(shape))
        self.ref = np.zeros(self.cells)
        self.m = np.zeros(self.cells, np.int32)
        self.sabs = np.zeros(self.cells)
        self.extra = None
        self.bad = 0

    def add(self, idx, w, delta=None):
        w = np.asarray(w, np.float64)
        live = w != 0 if delta is None else delta > 0        # NaN != 0: NaN weights count
        idx, w = idx[live], w[live]
        n = self.cells
        self.ref += np.bincount(idx, weights=w, minlength=n)
        self.m += np.bincount(idx, minlength=n).astype(np.int32)
        if delta is None:
            self.sabs += np.bincount(idx, weights=np.abs(w), minlength=n)
        else:
            d = delta[live]
            self.sabs += np.bincount(idx, weights=np.abs(w) + d, minlength=n)
            if self.extra is None:
                self.extra = np.zeros(n)
            self.extra += np.bincount(idx, weights=d, minlength=n)

    def done(self):
        for name in ("ref", "m", "sabs", "extra"):
            if getattr(self, name) is not None:
                setattr(self, name, getattr(self, name).reshape(self.shape))
        return self


def ref_int(events, bins, H, W, polarity):
    """torch_ref.events_to_voxel (event_utils.py) with float64 accumulation.  events [n,4] float32 or float64.  Events
    whose truncated pixel lies outside [-W,W) x [-H,H) (IndexError in the reference) are left out and counted in .bad;
    they still take part in the time normalisation, as they do in the kernel."""
    ev = np.asarray(events)
    f = ev.dtype.type
    g = _Grid((bins * (2 if polarity else 1), H, W))
    with np.errstate(invalid="ignore", divide="ignore"):
        xs, ys, ps = _trunc_i32(ev[:, 0]), _trunc_i32(ev[:, 1]), _trunc_i32(ev[:, 3])
        t = ev[:, 2]
        t = (t - t[0]) / ((t[-1] - t[0]) + 1e-6)
        tn = (t - t[0]) / (t[-1] - t[0]) * f(bins - 1)
        keep = (xs >= -W) & (xs < W) & (ys >= -H) & (ys < H)
        g.bad = int((~keep).sum())
        xs, ys, ps, tn = xs[keep], ys[keep], ps[keep], tn[keep]
        pix = np.where(ys < 0, ys + H, ys) * W + np.where(xs < 0, xs + W, xs)
        factors = [(ps > 0).astype(f), (ps <= 0).astype(f)] if polarity else [ps.astype(f)]
        for plane, fac in enumerate(factors):
            for b in range(bins):
                w = (fac * np.maximum(f(1.0) - np.abs(tn - f(b)), f(0))).astype(np.float32)
                delta = None
                if f is np.float64:
                    near = ~(np.abs(tn - b) >= 1 + 1e-5)                                  # NaN tn: near
                    delta = np.where(near, np.abs(fac) * (6 * bins + 3) * U, 0.0)
                g.add(pix + (plane * bins + b) * H * W, w, delta)
    return g.done()


def ref_trilinear(x, y, t, p, bins, H, W, polarity, taps=None):
    """torch_ref.events_to_voxel_trilinear (dsec.py) with float64 accumulation.  `taps`, if a list, receives for every
    (event, y tap, t tap) the kernel issues stores for: (plane, index of the left x tap in the grid, x0 valid, x0+1 valid)."""
    x, y = np.asarray(x, np.float32), np.asarray(y, np.float32)
    p, t = np.asarray(p).astype(np.float32), np.asarray(t, np.int64)
    g = _Grid((bins * (2 if polarity else 1), H, W))
    with np.errstate(invalid="ignore", divide="ignore"):
        ts = (t - t[0]).astype(np.float32)
        ts = ts / ts[-1]
        if polarity:
            subsets = [(p > 0, None), (p <= 0, np.float32(1))]
        else:
            subsets = [(np.ones(len(p), bool), None)]
        for plane, (sel, value) in enumerate(subsets):
            if not sel.any():
                continue
            xs, ys, tss = x[sel], y[sel], ts[sel]
            val = np.float32(2) * p[sel] - np.float32(1) if value is None else value
            tn = np.float32(bins - 1) * (tss - tss[0]) / (tss[-1] - tss[0])
            x0, y0, t0 = _trunc_i32(xs), _trunc_i32(ys), _trunc_i32(tn)
            for dx, dy, dt in itertools.product((0, 1), repeat=3):          # the reference's loop order
                xl, yl, tl = x0 + dx, y0 + dy, t0 + dt
                ok = (xl < W) & (xl >= 0) & (yl < H) & (yl >= 0) & (tl >= 0) & (tl < bins)
                w = (val * (1 - np.abs(xl.astype(np.float32) - xs)) * (1 - np.abs(yl.astype(np.float32) - ys))
                     * (1 - np.abs(tl.astype(np.float32) - tn)))
                lin = plane * bins * H * W + (tl * H + yl) * W + xl
                g.add(lin[ok], w[ok])
            if taps is not None:
                fin = (np.abs(xs) < 1e9) & (np.abs(ys) < 1e9) & (np.abs(tn) < 1e9)   # the kernel's own filter
                for dy, dt in itertools.product((0, 1), repeat=2):
                    yl, tl = y0 + dy, t0 + dt
                    v0, v1 = (x0 >= 0) & (x0 < W), (x0 + 1 >= 0) & (x0 + 1 < W)
                    ok = fin & (yl >= 0) & (yl < H) & (tl >= 0) & (tl < bins) & (v0 | v1)
                    cell = plane * bins * H * W + (tl * H + yl) * W + x0
                    taps.append((plane, cell[ok], v0[ok], v1[ok]))
    return g.done()


def check_cells(got, R, family, label, widen=True):
    """Hold an fp32 grid to reference R cell by cell (module docstring); returns the largest |got - ref| / bar."""
    got = np.asarray(got)
    assert got.dtype == np.float32 and got.shape == R.ref.shape, (got.dtype, got.shape, R.ref.shape)
    assert R.m.max() < 2 ** 14
    nan = np.isnan(R.ref)
    got_nan = np.isnan(got)
    assert np.array_equal(got_nan, nan), \
        f"{label}: NaN at {np.argwhere(got_nan & ~nan)[:5].tolist()} (not in ref), missing at {np.argwhere(nan & ~got_nan)[:5].tolist()}"
    extra = R.extra if (widen and R.extra is not None) else 0.0
    bar = np.maximum(R.m - 1, 0) * U * R.sabs * (1 + 2.0 ** -9) + extra
    empty = (R.m == 0) & ~nan
    nz = np.argwhere(empty & (got.view(np.uint32) != 0))
    assert nz.size == 0, f"{label}: cells with no contribution hold {got[tuple(nz[:5].T)]} at {nz[:5].tolist()}"
    diff = np.abs(got.astype(np.float64) - R.ref)
    with np.errstate(invalid="ignore"):
        over = ~nan & ~(diff <= bar)
    if over.any():
        at = np.argwhere(over)[:8]
        rows = [(c.tolist(), float(got[tuple(c)]), float(R.ref[tuple(c)]), int(R.m[tuple(c)]), float(np.asarray(bar)[tuple(c)]))
                for c in at]
        raise AssertionError(f"{label}: {int(over.sum())} cells over the bar; (cell, got, ref, m, bar): {rows}")
    live = ~nan & (bar > 0)
    ratio = float((diff[live] / bar[live]).max()) if live.any() else 0.0
    MEASURED[family] = max(MEASURED.get(family, 0.0), ratio)
    return ratio


@pytest.fixture(scope="module", autouse=True)
def _report_measured():
    yield
    if MEASURED:
        print("\nlargest |got - ref| / bar per case family:")
        for fam, v in sorted(MEASURED.items()):
            print(f"  {fam:24s} {v:.3g}")


# ------------------------------------------------------------------------------------------------- integer cases
def _rng(name):
    return np.random.default_rng(zlib.crc32(name.encode()))


def _ev(x, y, t, p, dtype=np.float32):
    return np.stack([np.asarray(a, np.float64) for a in (x, y, t, p)], 1).astype(dtype)


def _random_int(rng, n, H, W, bins, t0=0.0, span=1.0, p=(-1, 1)):
    t = t0 + np.sort(rng.random(n)) * span
    return dict(events=_ev(rng.integers(0, W, n), rng.integers(0, H, n), t, rng.choice(np.float32(p), n)),
                bins=bins, H=H, W=W)


def _int_tn(t, t_first, t_last, bins):
    """The reference's fp32 tn of stamps t for a window [t_first, t_last]."""
    t, tf, tl = np.float32(t), np.float32(t_first), np.float32(t_last)
    den = (tl - tf) + np.float32(1e-6)
    ts0, tsl = (tf - tf) / den, (tl - tf) / den
    return ((t - tf) / den - ts0) / (tsl - ts0) * np.float32(bins - 1)


def _int_tn_integer(rng):
    """bins = 5 and stamps tf + k (tl - tf) / 4: ts scales with dt by a power of two, so tn = k exactly (first and last
    event: 0 and bins - 1)."""
    bins, H, W, tf, tl = 5, 5, 8, 0.25, 1.25
    k = np.concatenate([[0], np.sort(rng.integers(0, bins, 200)), [bins - 1]])
    ts = np.float32(tf + (tl - tf) * k / (bins - 1))
    assert np.array_equal(_int_tn(ts, tf, tl, bins), k.astype(np.float32))
    n = len(ts)
    return dict(events=_ev(rng.integers(0, W, n), rng.integers(0, H, n), ts, rng.choice([-1, 1], n)), bins=bins, H=H, W=W)


def _int_unsorted(rng):
    c = _random_int(rng, 3000, 9, 11, 10, t0=2.0, span=3.0)
    ev = c["events"]
    ev[1:-1, 2] = 2.0 + (rng.random(len(ev) - 2) * 1.4 - 0.2) * 3.0      # interior: any order, 20 % outside the window
    return c


def _int_trunc_edges(rng):
    n, H, W = 2000, 6, 10
    fx = [lambda k: -rng.random(k) * 0.999, lambda k: np.full(k, W - 0.5), lambda k: rng.integers(0, W, k) + 0.75,
          lambda k: -W + 0.5 + np.zeros(k)]
    fy = [lambda k: -rng.random(k) * 0.999, lambda k: np.full(k, H - 0.5), lambda k: rng.integers(0, H, k) + 0.0]
    x = np.concatenate([f(n // 4) for f in fx])
    y = np.concatenate([fy[i % 3](1) for i in range(n)])
    c = _random_int(rng, n, H, W, 4)
    c["events"][:, 0], c["events"][:, 1] = x, y
    return c


def _int_wrap(rng):
    c = _random_int(rng, 2000, 7, 9, 5)
    c["events"][:, 0] = rng.integers(-9, 9, 2000)
    c["events"][:, 1] = rng.integers(-7, 7, 2000)
    return c


def _int_out_of_range(rng):
    c = _random_int(rng, 2000, 6, 8, 5)
    ev = c["events"]
    bad = rng.random(2000) < 0.1
    bad[[0, -1]] = False                                 # the window's ends stay in range
    ev[bad, 0] = rng.choice([-9, -20, 8, 9, 1e6], int(bad.sum()))
    more = ~bad & (rng.random(2000) < 0.05)
    more[[0, -1]] = False
    ev[more, 1] = rng.choice([-7, 6, 30], int(more.sum()))
    c["check_range"] = False
    return c


def _int_degenerate_burst(rng):
    n, H, W = 64, 5, 6
    return dict(events=_ev(rng.integers(-W, W, n), rng.integers(0, H, n), np.full(n, 3.5), rng.choice([-1, 0, 1, 2], n)),
                bins=4, H=H, W=W)


def _int_float64(rng):
    c = _random_int(rng, 3000, 12, 16, 10)
    ev = c["events"].astype(np.float64)
    ev[:, 2] = 1.6e9 + np.sort(rng.random(3000)) * 0.05                  # seconds since the epoch; fp32 ulp there is 128
    c["events"] = ev
    return c


INT_CASES = {
    "wrap_negative": _int_wrap,
    "trunc_edges": _int_trunc_edges,
    "tn_integer": _int_tn_integer,
    "unsorted": _int_unsorted,
    "p_values": lambda r: _random_int(r, 3000, 8, 12, 10, p=(-1, 0, 0.5, 1, 2)),
    "bins1": lambda r: _random_int(r, 1000, 5, 7, 1),
    "bins2": lambda r: _random_int(r, 1000, 5, 7, 2),
    "h1": lambda r: {**_random_int(r, 500, 1, 33, 3), "events": _ev(r.integers(-33, 33, 500), r.integers(-1, 1, 500),
                                                                   np.sort(r.random(500)), r.choice([-1, 1], 500))},
    "w1": lambda r: {**_random_int(r, 500, 17, 1, 3), "events": _ev(r.choice([0, -1, -0.5, 0.5], 500), r.integers(-17, 17, 500),
                                                                   np.sort(r.random(500)), r.choice([-1, 1], 500))},
    "float64": _int_float64,
    "out_of_range": _int_out_of_range,
    "degenerate_burst": _int_degenerate_burst,
    "degenerate_single": lambda r: dict(events=_ev([2], [1], [7.0], [-1]), bins=3, H=3, W=4),
    "degenerate_pair": lambda r: dict(events=np.float32([[1, 1, 0.5, 1], [2, 1, 0.5, -1]]), bins=3, H=3, W=4),
    "degenerate_bins1": lambda r: {**_int_degenerate_burst(r), "bins": 1},
    "things": lambda r: _random_int(r, 1_000_000, 540, 960, 10),
    "hd": lambda r: _random_int(r, 4_000_000, 1080, 1920, 10),
}
BIG = {"things", "hd", "dsec"}


@functools.lru_cache(maxsize=None)
def int_case(name):
    c = INT_CASES[name](_rng("int/" + name))
    c.setdefault("check_range", True)
    return c


@functools.lru_cache(maxsize=4)
def int_ref(name, polarity):
    c = int_case(name)
    return ref_int(c["events"], c["bins"], c["H"], c["W"], polarity)


# ------------------------------------------------------------------------------------------------- tri-linear cases
def _random_tri(rng, n, H, W, bins, t0=1_000_000, span=100_000):
    return dict(x=(rng.random(n) * (W - 1)).astype(np.float32), y=(rng.random(n) * (H - 1)).astype(np.float32),
                t=t0 + np.sort(rng.integers(0, span, n)), p=rng.integers(0, 2, n).astype(np.uint8), bins=bins, H=H, W=W)


def _tri_edges(rng, axis):
    H, W = (6, 10) if axis == "x" else (10, 7)
    c = _random_tri(rng, 2000, H, W, 4)
    L = W if axis == "x" else H
    r = rng.random(2000).astype(np.float32) * np.float32(0.999)
    v = np.select([np.arange(2000) % 4 == k for k in range(4)],
                  [-r, -1 - r, (L - 1) + r + np.float32(0.0005), L + r]).astype(np.float32)
    v[:8] = [-1, -0.0, L - 1, L, -2 + 2 ** -20, L - 2 ** -20, 0.5, -1.5]
    c[axis] = v
    return c


def _tri_tn_integer(rng):
    """Stamps at multiples of T/4 with bins = 5: tn = 0..4 exactly, in each polarity subset as in the whole window."""
    H, W, T, t0 = 6, 9, 4000, 1_000_000
    k = np.concatenate([[0, 0], rng.integers(0, 5, 400), [4, 4]])
    p = np.concatenate([[0, 1], rng.integers(0, 2, 400), [0, 1]]).astype(np.uint8)
    order = np.argsort(k, kind="stable")
    n = len(k)
    return dict(x=(rng.random(n) * (W - 1)).astype(np.float32), y=(rng.random(n) * (H - 1)).astype(np.float32),
                t=t0 + k[order] * (T // 4), p=p[order], bins=5, H=H, W=W)


def _tri_subset_one(rng):
    c = _random_tri(rng, 1000, 7, 9, 4)
    c["p"][:] = 0
    c["p"][500] = 1
    return c


def _tri_subset_same_time(rng):
    c = _random_tri(rng, 1000, 7, 9, 4)
    pos = c["p"] > 0
    c["t"] = np.where(pos, c["t"][500], c["t"])
    order = np.argsort(c["t"], kind="stable")
    for k in ("x", "y", "t", "p"):
        c[k] = c[k][order]
    return c


def _tri_nonfinite(rng):
    c = _random_tri(rng, 1200, 7, 9, 4)
    bad = np.float32([np.nan, np.inf, -np.inf, 1e30, -1e30, 1e9, -1e9, 2.5e9, -2.5e9, 2.0 ** 31, -2.0 ** 31, 2.1e9])
    i = rng.permutation(np.arange(1, 1199))[:600]
    c["x"][i[:300]] = bad[np.arange(300) % len(bad)]
    c["y"][i[300:]] = bad[np.arange(300) % len(bad)]
    return c


TRI_CASES = {
    "random": lambda r: _random_tri(r, 3000, 11, 13, 10),
    "integer_xy": lambda r: {**_random_tri(r, 1500, 9, 13, 5), "x": r.integers(0, 13, 1500).astype(np.float32),
                             "y": r.integers(0, 9, 1500).astype(np.float32)},
    "x_edges": lambda r: _tri_edges(r, "x"),
    "y_edges": lambda r: _tri_edges(r, "y"),
    "tn_integer": _tri_tn_integer,
    "subset_one": _tri_subset_one,
    "subset_same_time": _tri_subset_same_time,
    "all_positive": lambda r: {**_random_tri(r, 1000, 6, 8, 3), "p": np.ones(1000, np.uint8)},
    "all_negative": lambda r: {**_random_tri(r, 1000, 6, 8, 3), "p": np.zeros(1000, np.uint8)},
    "p_half": lambda r: {**_random_tri(r, 1500, 6, 8, 4), "p": r.choice(np.float32([0, 0.5, 1]), 1500)},
    "bins1": lambda r: _random_tri(r, 800, 5, 6, 1),
    "nonfinite_xy": _tri_nonfinite,
    "epoch_t": lambda r: _random_tri(r, 3000, 8, 10, 10, t0=1_600_000_000_000_000, span=50_000),
    "long_span": lambda r: _random_tri(r, 3000, 8, 10, 10, t0=1_600_000_000_000_000, span=300_000_000),
    "dsec": lambda r: _random_tri(r, 1_500_000, 480, 640, 10),
    "hd": lambda r: _random_tri(r, 4_000_000, 1080, 1920, 10),
}


def _census_case(rng, W):
    """Taps at the grid's first cell, at the last x pair (x0 = W - 2) of the last row of the last bin of both planes,
    at row ends and starts, plus random events; both subsets start and end at the window's ends."""
    H, bins, n = 5, 3, 300
    c = _random_tri(rng, n, H, W, bins)
    x, y, p = c["x"], c["y"], c["p"]
    x[:2], y[:2], p[:2] = 0.25, 0.25, [1, 0]
    x[-2:], y[-2:], p[-2:] = W - 1.5, H - 0.5, [1, 0]
    mid = np.arange(2, n - 2)
    x[mid[::3]] = W - 2 + rng.random(len(mid[::3])).astype(np.float32) * np.float32(0.99)
    x[mid[1::3]] = rng.random(len(mid[1::3])).astype(np.float32) * np.float32(0.99)
    return c


for _w in (12, 13, 14, 15):                              # W = 0, 1, 2, 3 (mod 4)
    TRI_CASES[f"census_w{_w}"] = functools.partial(_census_case, W=_w)


@functools.lru_cache(maxsize=None)
def tri_case(name):
    return TRI_CASES[name](_rng("tri/" + name))


@functools.lru_cache(maxsize=4)
def tri_ref(name, polarity):
    c = tri_case(name)
    return ref_trilinear(c["x"], c["y"], c["t"], c["p"], c["bins"], c["H"], c["W"], polarity)


def offsets(name):
    return {"things": (0,), "dsec": (0,), "hd": (1,)}.get(name, (0, 1, 2, 3))


SMALL_INT = [n for n in INT_CASES if n not in BIG]
SMALL_TRI = [n for n in TRI_CASES if n not in BIG]


# ------------------------------------------------------------------------------------------------- CPU checks
@pytest.mark.parametrize("polarity", [True, False])
@pytest.mark.parametrize("name", SMALL_INT)
def test_int_reference_matches_torch_ref(name, polarity):
    """The float64 reference against torch_ref's fp32 grid (index_put_ in event order), cell by cell."""
    c = int_case(name)
    ev = c["events"]
    R = int_ref(name, polarity)
    if not c["check_range"]:
        with pytest.raises(IndexError):
            torch_ref.events_to_voxel(ev, c["bins"], c["H"], c["W"], polarity)
        xs, ys = _trunc_i32(ev[:, 0]), _trunc_i32(ev[:, 1])
        ev = ev[(xs >= -c["W"]) & (xs < c["W"]) & (ys >= -c["H"]) & (ys < c["H"])]      # same first and last event
        assert R.bad == len(c["events"]) - len(ev) > 0
    with np.errstate(invalid="ignore"):
        want = torch_ref.events_to_voxel(ev, c["bins"], c["H"], c["W"], polarity)
    check_cells(want, R, "cpu torch_ref int", name, widen=False)
    if name.startswith("degenerate"):
        pix = np.isnan(R.ref).any(0)
        assert pix.any() and np.isnan(R.ref[:, pix]).all()                  # every channel at every event's pixel


@pytest.mark.parametrize("polarity", [True, False])
@pytest.mark.parametrize("name", SMALL_TRI)
def test_trilinear_reference_matches_torch_ref(name, polarity):
    c = tri_case(name)
    want = torch_ref.events_to_voxel_trilinear(c["x"], c["y"], c["t"], c["p"], c["bins"], c["H"], c["W"], polarity)
    check_cells(want, tri_ref(name, polarity), "cpu torch_ref trilinear", name)


@pytest.mark.parametrize("name,polarity", [("event_voxel_pol", True), ("event_voxel_nopol", False),
                                           ("event_trilinear_pol", True), ("event_trilinear_nopol", False)])
def test_reference_matches_upstream_fixtures(golden, name, polarity):
    g = golden(name)
    bins, H, W = int(g["bins"]), int(g["H"]), int(g["W"])
    if "events" in g:
        R = ref_int(g["events"], bins, H, W, polarity)
    else:
        R = ref_trilinear(g["x"], g["y"], g["t"], g["p"], bins, H, W, polarity)
    check_cells(g["vox"], R, "cpu upstream fixtures", name)


@pytest.mark.parametrize("polarity", [True, False])
def test_oracle_agrees_with_the_reference(polarity):
    """oracle/spec.c (fp32, event order) on every small case, the zero-length windows included."""
    from oracle import spec
    for name in SMALL_INT:
        c = int_case(name)
        vox, bad = spec.event_voxel_int(c["events"].astype(np.float32) if name != "float64" else _shifted(c["events"]),
                                        c["bins"], c["H"], c["W"], polarity)
        R = int_ref(name, polarity)
        assert bad == R.bad, name
        check_cells(vox, R, "cpu oracle int", name)
    for name in SMALL_TRI:
        c = tri_case(name)
        vox = spec.event_voxel_trilinear(c["x"], c["y"], c["t"], c["p"], c["bins"], c["H"], c["W"], polarity)
        check_cells(vox, tri_ref(name, polarity), "cpu oracle trilinear", name)


def _shifted(ev64):
    """What eventsToVoxel hands the kernel for a float64 array (events.py): stamps shifted in float64, then cast."""
    ev = ev64.astype(np.float32)
    ev[:, 2] = ev64[:, 2] - ev64[0, 2]
    return ev


STORE = ("v2", "v4", "scalar")


def store_census(names):
    """Which store each tap of the tri-linear kernel issues, over the cases and `out` offsets the GPU tests run."""
    seen, flags = set(), set()
    for name in names:
        c = tri_case(name)
        H, W, bins = c["H"], c["W"], c["bins"]
        for polarity in (True, False):
            taps = []
            ref_trilinear(c["x"], c["y"], c["t"], c["p"], bins, H, W, polarity, taps=taps)
            total = bins * (2 if polarity else 1) * H * W
            for off in offsets(name):
                for plane, cell, v0, v1 in taps:
                    a = (off + cell) % 4                           # float slot in its 16-byte group
                    both = v0 & v1
                    v2 = both & (a % 2 == 0)
                    v4 = both & (a == 1) & (cell > 0) & (cell + 2 < total)
                    path = np.where(v2, 0, np.where(v4, 1, 2))
                    for k in np.unique(path):
                        seen.add((STORE[k], plane, off))
                    x0 = cell % W
                    if (both & (a == 1) & (cell == 0)).any():
                        flags.add("first cell: v4 refused")
                    if (both & (a == 1) & (cell + 2 == total)).any():
                        flags.add("last pair: v4 refused")
                    if (v4 & (x0 == W - 2) & ((cell + 2) % (bins * H * W) != 0)).any():
                        flags.add("v4 across a row end")
                    if (v4 & (x0 == 0)).any():
                        flags.add("v4 across a row start")
                    if polarity and (v4 & ((cell + 2 == bins * H * W) | (cell == bins * H * W))).any():
                        flags.add("v4 across the polarity planes")
    return seen, flags


def test_store_paths_are_all_reached():
    seen, flags = store_census(SMALL_TRI)
    for path in STORE:
        for plane in (0, 1):
            for off in range(4):
                assert (path, plane, off) in seen, (path, plane, off)
    assert flags == {"first cell: v4 refused", "last pair: v4 refused", "v4 across a row end", "v4 across a row start",
                     "v4 across the polarity planes"}, flags


# ------------------------------------------------------------------------------------------------- GPU
DEV = torch.device("cuda", 0)


def _poisoned(shape, off):
    """`out` of `shape` starting `off` floats past a 16-byte boundary of a NaN-poisoned buffer with 64-float guards."""
    cells = int(np.prod(shape))
    buf = torch.full((64 + off + cells + 64,), POISON, dtype=torch.int32, device=DEV)
    assert buf.data_ptr() % 16 == 0
    return buf, buf[64 + off:64 + off + cells].view(torch.float32).view(shape)


def _collect(buf, off, shape, label):
    torch.cuda.synchronize()
    bits = buf.cpu().numpy()
    cells = int(np.prod(shape))
    inside = bits[64 + off:64 + off + cells]
    assert (bits[:64 + off] == POISON).all() and (bits[64 + off + cells:] == POISON).all(), f"{label}: wrote outside `out`"
    assert (inside != POISON).all(), f"{label}: {int((inside == POISON).sum())} floats of `out` not written"
    return inside.view(np.float32).reshape(shape)


def run_int(ev32, bins, H, W, polarity, check_range, off):
    from rpeflow_b200.events import events_to_voxel_device
    shape = (bins * (2 if polarity else 1), H, W)
    buf, out = _poisoned(shape, off)
    got = events_to_voxel_device(torch.from_numpy(ev32).to(DEV), bins, H, W, polarity, check_range=check_range, out=out)
    assert got.data_ptr() == out.data_ptr()
    return _collect(buf, off, shape, f"off {off}")


def run_trilinear(c, polarity, off):
    from rpeflow_b200.events import events_to_voxel_trilinear_device
    shape = (c["bins"] * (2 if polarity else 1), c["H"], c["W"])
    buf, out = _poisoned(shape, off)
    x, y, t, p = (torch.from_numpy(np.asarray(c[k])).to(DEV) for k in ("x", "y", "t", "p"))
    events_to_voxel_trilinear_device(x, y, t, p, c["bins"], c["H"], c["W"], polarity, out=out)
    return _collect(buf, off, shape, f"off {off}")


@pytest.mark.gpu
@pytest.mark.parametrize("polarity", [True, False])
@pytest.mark.parametrize("name", [n for n in INT_CASES if n != "float64"])
def test_int_voxeliser_vs_float64(name, polarity):
    c = int_case(name)
    R = int_ref(name, polarity)
    family = "int " + ("degenerate" if name.startswith("degenerate") else name if name in BIG else "small")
    if not c["check_range"]:
        with pytest.raises(IndexError):
            run_int(c["events"], c["bins"], c["H"], c["W"], polarity, True, 0)
    for off in offsets(name):
        got = run_int(c["events"], c["bins"], c["H"], c["W"], polarity, c["check_range"], off)
        check_cells(got, R, family, f"{name} off {off}")


@pytest.mark.gpu
@pytest.mark.parametrize("polarity", [True, False])
def test_int_voxeliser_float64_events(polarity):
    """float64 arrays go through eventsToVoxel's float64 shift; the reference keeps its float64 weights."""
    import rpeflow_b200 as b200
    c = int_case("float64")
    got = b200.eventsToVoxel(c["events"], num_bins=c["bins"], height=c["H"], width=c["W"], event_polarity=polarity)
    check_cells(got, int_ref("float64", polarity), "int float64", "float64")


@pytest.mark.gpu
@pytest.mark.parametrize("polarity", [True, False])
@pytest.mark.parametrize("name", list(TRI_CASES))
def test_trilinear_voxeliser_vs_float64(name, polarity):
    c = tri_case(name)
    R = tri_ref(name, polarity)
    family = "trilinear " + (name if name in BIG else "census" if name.startswith("census") else "small")
    for off in offsets(name):
        check_cells(run_trilinear(c, polarity, off), R, family, f"{name} off {off}")


# ------------------------------------------------------------------------------------------------- the bench's batched path
@functools.lru_cache(maxsize=1)
def _stack_inputs(name, batch):
    from rpeflow_b200.stack import CONFIGS, make_host_inputs
    cfg = CONFIGS[name]
    host = make_host_inputs(cfg, batch)
    if name == "dsec":
        refs = [ref_trilinear(host["ev_x"][i].numpy(), host["ev_y"][i].numpy(), host["ev_t"][i].numpy(),
                              host["ev_p"][i].numpy(), cfg.event_bins, cfg.height, cfg.width, True) for i in range(batch)]
    else:
        refs = [ref_int(host["events"][i].numpy(), cfg.event_bins, cfg.height, cfg.width, True) for i in range(batch)]
    return cfg, host, refs


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["dsec", "things"])
def test_stack_voxelise_every_sample(name):
    """CostVolumeStack.voxelise at batch 3: each sample writes its slice grids[i] of one batched tensor, dealt onto one
    side stream or two (samples 0 and 2 then share a lane).  Every sample against its reference."""
    from rpeflow_b200.stack import CostVolumeStack, to_device
    cfg, host, refs = _stack_inputs(name, 3)
    stack = CostVolumeStack(cfg, DEV)
    x = to_device(host, DEV)
    for lanes in (2, 1):
        grids = stack.voxelise(x, lanes=lanes)
        torch.cuda.synchronize()
        for i, R in enumerate(refs):
            check_cells(grids[i].cpu().numpy(), R, f"batched {name}", f"{name} lanes {lanes} sample {i}")


@pytest.mark.gpu
def test_graph_replay_voxels_every_sample():
    """One replay of the fused CUDA graph of the whole DSEC stack at batch 3: its voxel grids against the reference."""
    from rpeflow_b200.stack import CostVolumeStack, GraphedStack, to_device
    cfg, host, refs = _stack_inputs("dsec", 3)
    stack = CostVolumeStack(cfg, DEV)
    assert stack.voxel_lanes == 2
    g = GraphedStack(stack, to_device(host, DEV), fused=True, with_checksum=False)
    g.out["event_voxel"].fill_(float("nan"))
    out = g.replay()
    torch.cuda.synchronize()
    for i, R in enumerate(refs):
        check_cells(out["event_voxel"][i].cpu().numpy(), R, "batched dsec graph", f"graph sample {i}")
