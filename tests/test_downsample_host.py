"""CPU tests of equal-depth subsampling (DESIGN S0d): the read-by-read reference (tests/downsample_oracle.py), the
host logic of LoadedGenome.downsample / equal_depth on a stand-in genome, the C ABI symbols and the R routines'
argument checks under the stand-in R runtime of tests/mock_r."""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest

from tadpole_b200 import _lib
from tadpole_b200.batch import LoadedGenome, _CtxRef, equal_depth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import downsample_oracle as G  # noqa: E402


def _genome(seed=0):
    rng = np.random.default_rng(seed)
    sizes = [30, 1, 20]
    starts = np.concatenate(([0], np.cumsum(sizes)))
    b1, b2, v = [], [], []
    for c, n in enumerate(sizes):
        for _ in range(60):
            i = int(rng.integers(0, n)); j = min(n - 1, i + int(rng.integers(0, 5)))
            b1.append(starts[c] + i); b2.append(starts[c] + j); v.append(float(rng.integers(0, 40)))
    b1 += [3, 40]; b2 += [35, 31]; v += [5.0, 7.0]                   # a trans pixel and one below the diagonal
    return sizes, np.array(b1), np.array(b2), np.array(v)


def _kept(out):
    return [dict(zip(zip(i.tolist(), j.tolist()), k.tolist())) for i, j, k in out]


def test_oracle_keeps_exactly_n_reads_and_no_cell_more_than_it_had():
    sizes, b1, b2, v = _genome()
    c, i, j, n = G.merged_cells(sizes, b1, b2, v)
    have = {(int(a), int(b), int(x)): int(y) for a, b, x, y in zip(c, i, j, n)}
    total = int(n.sum())
    for N in (0, 1, total // 3, total - 1, total):
        out = G.downsample(sizes, b1, b2, v, N, seed=5)
        assert sum(int(k.sum()) for _, _, k in out) == N
        for ch, d in enumerate(_kept(out)):
            for (a, b), k in d.items():
                assert 0 < k <= have[(ch, a, b)]
    assert all(i.size == 0 for i, _, _ in G.downsample(sizes, b1, b2, v, 0, seed=5))
    with pytest.raises(ValueError, match="contacts asked for"):
        G.downsample(sizes, b1, b2, v, total + 1, seed=0)


def test_oracle_ignores_pixel_order_and_duplicate_splitting():
    sizes, b1, b2, v = _genome(1)
    total = int(G.merged_cells(sizes, b1, b2, v)[3].sum())
    N = total // 2
    ref = _kept(G.downsample(sizes, b1, b2, v, N, seed=2 ** 40 + 3))
    perm = np.random.default_rng(9).permutation(v.size)
    assert _kept(G.downsample(sizes, b1[perm], b2[perm], v[perm], N, seed=2 ** 40 + 3)) == ref
    # every count split into two entries (one of them possibly 0)
    part = np.floor(v / 3)
    sb1, sb2, sv = np.concatenate((b1, b1)), np.concatenate((b2, b2)), np.concatenate((part, v - part))
    assert _kept(G.downsample(sizes, sb1, sb2, sv, N, seed=2 ** 40 + 3)) == ref
    # N = T gives the merged input back
    c, i, j, n = G.merged_cells(sizes, b1, b2, v)
    full = _kept(G.downsample(sizes, b1, b2, v, total, seed=1))
    assert full == [{(int(a), int(b)): float(x) for a, b, x in zip(i[c == ch], j[c == ch], n[c == ch])}
                    for ch in range(len(sizes))]
    assert _kept(G.downsample(sizes, b1, b2, v, N, seed=4)) != ref


def test_oracle_rejects_non_integer_and_oversized_cells():
    with pytest.raises(ValueError, match=r"chromosome 0, bins \(1, 2\): count 2.5"):
        G.downsample([4], [0, 1], [0, 2], [1.0, 2.5], 1, 0)
    with pytest.raises(ValueError, match="not an integer"):
        G.downsample([4], [0], [0], [-1.0], 0, 0)
    with pytest.raises(ValueError, match=r"bins \(3, 3\): the cell adds up to 2\^32"):
        G.downsample([4], [0, 3, 3], [0, 3, 3], [1.0, 2.0 ** 31, 2.0 ** 31], 1, 0)


def test_oracle_draws_the_hypergeometric_distribution():
    # cells of 3 and 2 reads, N = 2: P(kept = (2, 0), (1, 1), (0, 2)) = (3, 6, 1) / C(5, 2)
    nseed = 20000
    freq = np.zeros(3)
    for s in range(nseed):
        d = _kept(G.downsample([4], [0, 1], [0, 1], [3.0, 2.0], 2, s))[0]
        freq[2 - int(d.get((0, 0), 0))] += 1
    freq /= nseed
    p = np.array([0.3, 0.6, 0.1])
    # each frequency within 5 binomial standard deviations (a false alarm has probability below 2e-6 per entry)
    assert np.all(np.abs(freq - p) <= 5 * np.sqrt(p * (1 - p) / nseed)), freq


# ---- host logic on a stand-in genome --------------------------------------------------------------------------------

class _FakeGenome:
    def __init__(self, depth, log):
        self.chrom_bins = np.array([10, 5], dtype=np.int32)
        self._depth = np.array(depth, dtype=np.uint64)
        self.log, self.closed = log, False

    def depth(self):
        return self._depth

    def downsample(self, contacts, seed):
        self.log.append((int(self._depth.sum()), contacts, seed))
        return _FakeGenome([contacts, 0], self.log)

    def pixels(self, chrom):
        return np.array([3, 0, 0], np.int32), np.array([4, 2, 1], np.int32), np.array([1.0, 2.0, 3.0])

    def stats(self):
        return self._depth.astype(np.int64), 0, 0

    def close(self):
        self.closed = True


class _FakeCtx:
    closed = False

    def close(self):
        self.closed = True


def _loaded(depth, log, ctx=None, own=True):
    return LoadedGenome(_FakeGenome(depth, log), ["chrA", "chrB"], _CtxRef(ctx or _FakeCtx(), own))


def test_depth_fraction_and_argument_errors():
    log = []
    g = _loaded([7, 4], log)
    assert g.depth() == {"chrA": 7, "chrB": 4} and g.total_depth == 11
    g.downsample(fraction=0.5)
    g.downsample(fraction=1 / 3, seed=2 ** 64 + 5)
    g.downsample(contacts=11, seed=-1)
    g.downsample(fraction=0.0)
    assert log == [(11, 5, 0), (11, 3, 5), (11, 11, 2 ** 64 - 1), (11, 0, 0)]
    assert math.floor(0.5 * 11) == 5
    for kw, msg in ((dict(), "exactly one"), (dict(contacts=3, fraction=0.1), "exactly one"),
                    (dict(contacts=12), r"0\.\.11"), (dict(contacts=-1), r"0\.\.11"), (dict(fraction=1.5), r"\[0, 1\]")):
        with pytest.raises(ValueError, match=msg):
            g.downsample(**kw)
    i, j, v = g.pixels("chrB")
    assert i.tolist() == [0, 0, 3] and j.tolist() == [1, 2, 4] and v.tolist() == [3.0, 2.0, 1.0]
    with pytest.raises(ValueError, match="unknown chromosome"):
        g.pixels("chrZ")


def test_equal_depth_subsamples_every_deeper_genome_with_its_own_seed():
    log = []
    a, b, c = _loaded([50, 10], log), _loaded([20, 5], log), _loaded([30, 0], log)
    out = equal_depth(a, b, c, seed=7)
    assert out[1] is b
    assert log == [(60, 25, 7), (30, 25, 9)]
    assert [g.total_depth for g in out] == [25, 25, 25]
    same = equal_depth(b, b)
    assert same[0] is b and same[1] is b


def test_the_context_is_closed_with_the_last_genome_that_uses_it():
    log = []
    ctx = _FakeCtx()
    g = _loaded([5, 5], log, ctx)
    sub = g.downsample(contacts=4)
    g.close()
    assert not ctx.closed and g._g is None
    with sub:
        pass
    assert ctx.closed and sub._g is None
    given = _FakeCtx()
    with _loaded([1, 1], log, given, own=False):
        pass
    assert not given.closed


# ---- ABI and R ------------------------------------------------------------------------------------------------------

def test_new_symbols_are_declared_and_bound():
    with open(os.path.join(ROOT, "include", "tadpole_b200.h")) as fh:
        header = fh.read()
    for name in ("tp_genome_depth", "tp_genome_downsample", "tp_genome_pixels"):
        assert re.search(r"\bint %s\(" % name, header), name
        assert name in _lib.EXPORTED
    lib = _lib.load()
    assert lib.tp_version() >= 107
    out = ctypes.c_void_p()
    assert lib.tp_genome_downsample(None, None, 1, 0, ctypes.byref(out)) == _lib.TP_ERR_ARG
    assert "null argument" in lib.tp_last_error().decode()
    reads = (ctypes.c_ulonglong * 1)()
    assert lib.tp_genome_depth(None, None, reads) == _lib.TP_ERR_ARG
    assert lib.tp_genome_pixels(None, None, 0, None, None, None) == _lib.TP_ERR_ARG


@pytest.fixture(scope="module")
def R():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import __graft_entry__ as g
    g.build()
    from mock_r.driver import MockR
    r = MockR()
    yield r
    r.reset()


def test_r_routines_are_registered_and_check_their_arguments(R):
    from mock_r.driver import RError
    for name, nargs in (("C_tp_genome_depth", 3), ("C_tp_genome_downsample", 5), ("C_tp_genome_pixels", 4)):
        assert R.registered(name) == nargs
        with pytest.raises(RError, match=f"takes {nargs} arguments"):
            R.call(name, *([0] * (nargs - 1)))
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_genome_depth", 0, 0, 1)
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_genome_downsample", 0, 0, 1, 1.0, 0.0)
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_genome_pixels", 0, 0, 0, 1)
