"""Read-level network at the edges of its device tiling, against the CPU oracle (oracle/rl_oracle.py, itself pinned to the
reference's class by tests/test_read_level.py::test_oracle_matches_reference_class).

  * full 16-window tiles of the tensor-core LSTM over recurrences of 1000-4000 steps;
  * the benched shape (256 windows x 1000 positions x 30 reads);
  * properties that need no oracle: a window's output does not depend on its batch mates, its slot or how the batch is
    split into device calls (bit for bit: no reduction crosses windows), and a window without reads (NaN) leaves the
    other windows of its LSTM tile bit-identical;
  * the order of the reads, empty ones in the middle included, only moves the result by summation order;
  * the fp32 convolution with more than 65 535 (window, read) rows in one call.

Every case runs all four (convolution, LSTM) pairs of tensor-core / fp32 kernels unless it says otherwise.  Bar as in
tests/test_read_level.py: probabilities within 2e-5 absolute, labels identical where the oracle's top-2 margin exceeds 1e-4.
The CPU oracle runs on subsets of windows where the batch is large.
"""
import functools

import numpy as np
import pytest

from oracle import rl_oracle

pytestmark = pytest.mark.gpu

TOL = 2e-5
PAIRS = {"tc": (True, True), "fp32": (False, False), "tc_lstm32": (True, False), "fp32_lstmtc": (False, True)}
SEED = 31


def features(B, P, D, seed, empty_rows=2, p_gap=0.15):
    """Read-level features int8 [B, P, D, 4], vectorised for large batches: reads cover a random span of the window,
    up to ``empty_rows`` trailing reads are empty (collate padding) and a fraction ``p_gap`` of the others are empty
    too (reads of the region that do not reach this window).  Every window has at least one read."""
    rs = np.random.RandomState(seed)
    lo = rs.randint(0, max(1, P // 3), (B, 1, D))
    hi = P - rs.randint(0, max(1, P // 3), (B, 1, D))
    p = np.arange(P)[None, :, None]
    depth = D - rs.randint(0, empty_rows + 1, (B, 1, 1))
    present = (np.arange(D)[None, None, :] < depth) & (rs.uniform(size=(B, 1, D)) >= p_gap)
    present[..., 0] |= ~present.any(-1)                      # every window keeps at least one read
    cover = (p >= lo) & (p < hi) & present
    base = rs.choice(5, size=(B, P, D), p=[0.23, 0.23, 0.23, 0.23, 0.08]) + 1
    qual = np.where(base == 5, 0, rs.randint(1, 55, (B, P, D)))
    strand = np.broadcast_to(rs.randint(0, 2, (B, 1, D)), (B, P, D))
    mapq = np.broadcast_to(rs.randint(1, 61, (B, 1, D)), (B, P, D))
    x = np.stack([base, qual, strand, mapq], -1) * cover[..., None]
    return x.astype(np.int8)


@functools.lru_cache(maxsize=None)
def _state_dict():
    return rl_oracle.synth_rl_state_dict(SEED)


@functools.lru_cache(maxsize=None)
def _oracle():
    return rl_oracle.build(_state_dict())


def _forward(x, pair, max_cells=None):
    from medaka_b200 import read_level
    m = read_level.LatentSpaceLSTM()
    m.load_state_dict(_state_dict())
    m.set_conv(*PAIRS[pair])
    if max_cells is not None:
        m.max_cells = max_cells
    try:
        return m.forward_arrays(x)
    finally:
        m.close()


def _check(label, got, want):
    err = float(np.abs(got - want).max())
    print("%s: max abs err %.2e" % (label, err))
    assert got.shape == want.shape and np.isfinite(got).all()
    assert err < TOL, err
    top2 = np.sort(want, -1)[..., -2:]
    decided = (top2[..., 1] - top2[..., 0]) > 1e-4
    assert np.array_equal(np.argmax(got, -1)[decided], np.argmax(want, -1)[decided])


# ------------------------------------------------------------------ full LSTM tiles, long recurrences
TILE_SHAPES = [(16, 4000, 3), (32, 2000, 4), (33, 1000, 6), (48, 1500, 3)]


@functools.lru_cache(maxsize=None)
def _tile_case(B, P, D):
    x = features(B, P, D, seed=B * 7 + P)
    return x, rl_oracle.predict(_oracle(), x)


@pytest.mark.parametrize("pair", list(PAIRS))
@pytest.mark.parametrize("B,P,D", TILE_SHAPES)
def test_full_lstm_tiles_long_recurrence(B, P, D, pair):
    """16 windows per tensor-core LSTM CTA: one, two and three full tiles, and two full tiles plus one window."""
    x, want = _tile_case(B, P, D)
    _check("%dx%dx%d/%s" % (B, P, D, pair), _forward(x, pair), want)


# ------------------------------------------------------------------ the benched shape and window independence
BENCH = (256, 1000, 30)
SPREAD = np.linspace(0, BENCH[0] - 1, 16).astype(int)


@functools.lru_cache(maxsize=None)
def _bench_x():
    return features(*BENCH, seed=5)


@functools.lru_cache(maxsize=None)
def _bench_out(pair):
    return _forward(_bench_x(), pair)


def test_benched_shape_spread_windows():
    x = _bench_x()
    want = rl_oracle.predict(_oracle(), x[SPREAD])
    _check("%dx%dx%d windows %s" % (BENCH + (SPREAD.tolist(),)), _bench_out("tc")[SPREAD], want)


@pytest.mark.parametrize("pair", ["tc", "fp32"])
def test_window_independence_and_call_splitting(pair):
    """A window's probabilities do not depend on its batch mates, its slot in the LSTM tile or the split into device
    calls: no reduction crosses windows, so the results are bit-identical."""
    x, full = _bench_x(), _bench_out(pair)
    idx = np.random.RandomState(2).permutation(BENCH[0])[:77]
    sub = _forward(np.ascontiguousarray(x[idx]), pair)
    assert np.array_equal(sub, full[idx]), np.abs(sub - full[idx]).max()
    split = _forward(x, pair, max_cells=BENCH[1] * BENCH[2] * 37)        # calls of 37, ..., 37, 34 windows
    assert np.array_equal(split, full), np.abs(split - full).max()


# ------------------------------------------------------------------ a window without reads
@pytest.mark.parametrize("pair", list(PAIRS))
def test_empty_window_leaves_tile_mates_unchanged(pair):
    """The window without reads is NaN (0 / 0 in the mean over reads, like the reference); the 15 others of its
    16-window LSTM tile are bit-identical to the batch without it."""
    x = features(15, 300, 10, seed=8)
    with_empty = np.insert(x, 6, 0, axis=0)
    base, got = _forward(x, pair), _forward(with_empty, pair)
    assert np.isnan(got[6]).all()
    mates = np.delete(got, 6, 0)
    assert np.array_equal(mates, base), np.abs(mates - base).max()
    _check("15 windows + empty/%s vs oracle" % pair, base[:4], rl_oracle.predict(_oracle(), x[:4]))


# ------------------------------------------------------------------ read order
@pytest.mark.parametrize("pair", list(PAIRS))
def test_read_order(pair):
    """Permuting the reads (empty ones in the middle of the window included) regroups them into other groups of 4 and
    other pairs; only the summation order changes."""
    x = features(4, 300, 14, seed=9, empty_rows=3, p_gap=0.3)
    empty = ~x.any((1, 3))
    assert empty[:, :-3].any()                               # interior empties exist before the permutation
    perm = np.random.RandomState(4).permutation(x.shape[2])
    want = rl_oracle.predict(_oracle(), x)
    _check("read order/%s" % pair, _forward(np.ascontiguousarray(x[:, :, perm]), pair), want)


# ------------------------------------------------------------------ fp32 convolution beyond 65 535 reads per call
def test_fp32_convolution_many_reads_per_call():
    """700 windows x 100 reads = 70 000 (window, read) rows in one call (the default max_cells keeps the batch whole)."""
    B, P, D = 700, 20, 100
    x = features(B, P, D, seed=10, empty_rows=5)
    fp32 = _forward(x, "fp32")
    sub = np.array([0, 1, 350, 654, 655, 656, 698, 699])
    _check("%dx%dx%d fp32 windows %s vs oracle" % (B, P, D, sub.tolist()), fp32[sub], rl_oracle.predict(_oracle(), x[sub]))
    _check("%dx%dx%d fp32 vs tc" % (B, P, D), fp32, _forward(x, "tc"))
