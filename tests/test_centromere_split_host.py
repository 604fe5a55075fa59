"""CPU tests of tp_centromere_split, load_mat's centromere split (R/TADpole.R:58-86) in the library: against a literal
restatement of the reference kept here (the numpy code api._split_centromere ran before the split moved into the
library), with and without the repair of quirk Q3, through the ctypes binding, api._split_centromere and the R shim."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def split_reference(bad, fix=False):
    """R/TADpole.R:58-86: None when there is no bad bin; else (cs, ce, None) when the longest run touches an end, or
    (cs, ce, ((keep_p, bad_p), (keep_q, bad_q))) with keep 0-based and bad columns original 1-based or None."""
    n = bad.size
    idx = np.flatnonzero(bad) + 1
    if idx.size == 0:
        return None
    brk = np.flatnonzero(np.diff(idx) > 1) + 1
    runs = np.split(idx, brk)
    longest = runs[int(np.argmax([len(r) for r in runs]))]       # which.max: first on ties
    cs, ce = int(longest[0]), int(longest[-1])
    if cs == 1 or ce == n:
        return cs, ce, None
    idx_p = np.arange(1, cs)
    idx_q = np.arange(ce + 1, n + 1)
    bad_p = idx[idx < cs]
    bad_q = idx[idx > ce]
    keep_p = np.ones(idx_p.size, bool)
    keep_p[bad_p - 1] = False
    keep_q = np.ones(idx_q.size, bool)
    if fix:
        keep_q[bad_q - ce - 1] = False
    else:
        inr = bad_q[bad_q <= idx_q.size]                           # quirk Q3
        keep_q[inr - 1] = False
    return cs, ce, ((idx_p[keep_p] - 1, bad_p if bad_p.size else None), (idx_q[keep_q] - 1, bad_q if bad_q.size else None))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from tadpole_b200 import _lib
    return _lib


def same_arm(got, want):
    (kg, bg), (kw, bw) = got, want
    assert kg.tolist() == kw.tolist()
    assert (bg is None) == (bw is None)
    if bw is not None:
        assert bg.tolist() == bw.tolist()


def check(lib, bad, fix):
    want = split_reference(bad, fix)
    split, span, p, q = lib.centromere_split(bad, fix)
    if want is None:
        assert not split and span is None and p is None and q is None
        return want
    assert span == want[:2]
    assert split == (want[2] is not None)
    if split:
        same_arm(p, want[2][0])
        same_arm(q, want[2][1])
    return want


def edge_cases():
    n = 40
    out = []
    out.append(np.zeros(n, bool))                                  # no bad bins
    one = np.zeros(n, bool); one[17] = True; out.append(one)       # one bad bin
    first = np.zeros(n, bool); first[:5] = True; first[20:22] = True; out.append(first)    # longest run at bin 1
    last = np.zeros(n, bool); last[-6:] = True; last[10] = True; out.append(last)         # longest run at bin n
    tie = np.zeros(n, bool); tie[8:11] = True; tie[25:28] = True; out.append(tie)         # two longest runs
    # q-arm bad columns inside and beyond the arm's length (Q3): centromere at 6..9, q arm 10..40 (31 bins)
    q3 = np.zeros(n, bool); q3[5:9] = True; q3[[2, 13, 29, 36]] = True; out.append(q3)
    out.append(np.ones(n, bool))                                   # every bin bad
    out.append(np.array([False, True, False]))                     # the smallest split
    return out


@pytest.mark.parametrize("fix", [False, True])
def test_split_matches_reference_on_edge_cases(lib, fix):
    results = [check(lib, b, fix) for b in edge_cases()]
    assert results[0] is None
    assert results[1][2] is not None and results[1][:2] == (18, 18)
    assert results[2][:2] == (1, 5) and results[2][2] is None
    assert results[3][:2] == (35, 40) and results[3][2] is None
    assert results[4][:2] == (9, 11)                               # the first of the tied runs
    (kq, bq) = results[5][2][1]
    assert bq.tolist() == [14, 30, 37]
    # Q3: 14 <= 31 and 30 <= 31 drop the q arm's 14th and 30th rows, 37 is ignored; fixed: the bad columns themselves
    assert (13 not in kq) == fix and (9 + 13 not in kq) == (not fix) and (36 not in kq) == fix


@pytest.mark.parametrize("fix", [False, True])
def test_split_matches_reference_on_random_flags(lib, fix):
    rng = np.random.default_rng(3 + fix)
    for t in range(3000):
        n = int(rng.integers(1, 120))
        bad = rng.random(n) < rng.choice([0.02, 0.1, 0.3, 0.6])
        if t % 3 == 0 and n > 8:                                  # a run that plays the centromere
            c0 = int(rng.integers(0, n - 3))
            bad[c0: c0 + int(rng.integers(1, 8))] = True
        check(lib, bad, fix)


def test_api_wrapper_keeps_its_return_value(lib, capsys):
    from tadpole_b200 import api
    rng = np.random.default_rng(5)
    was = api.QUIET
    api.QUIET = False
    try:
        for b in edge_cases()[1:] + [rng.random(300) < 0.05 for _ in range(50)]:
            if not b.any():
                continue
            for fix in (False, True):
                want = split_reference(b, fix)
                got = api._split_centromere(b, fix)
                lines = capsys.readouterr().err.splitlines()
                assert lines[0] == f"centromere position: {want[0]} {want[1]}"
                if want[2] is None:
                    assert got is None and lines[1:] == ["longest stretch of bad rows/columns at the ends, not splitting the matrix."]
                    continue
                assert len(lines) == 1
                (kp, bp), (kq, bq), cen = got
                same_arm((kp, bp), want[2][0])
                same_arm((kq, bq), want[2][1])
                assert cen.tolist() == list(range(want[0], want[1] + 1))
    finally:
        api.QUIET = was


def test_r_shim_split_gives_the_same_lists(lib):
    from mock_r.driver import MockR
    R = MockR()
    try:
        rng = np.random.default_rng(9)
        for b in edge_cases() + [rng.random(200) < 0.05 for _ in range(40)]:
            for fix in (False, True):
                head, kp, bp, kq, bq = R.call("C_tp_split", b.astype(np.int32), fix)
                split, span, p, q = lib.centromere_split(b, fix)
                assert head.tolist() == [int(split), *(span or (0, 0))]
                if not split:
                    assert kp is None and bp is None and kq is None and bq is None
                    continue
                for (k, bc), (kw, bw) in (((kp, bp), p), ((kq, bq), q)):
                    assert k.tolist() == (kw + 1).tolist()                 # R: 1-based keep
                    assert (bc is None) == (bw is None) and (bw is None or bc.tolist() == bw.tolist())
    finally:
        R.reset()
