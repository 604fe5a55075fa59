"""The score matrix is as wide as the largest level count, known only after the sweep.  With a small level_cap the CH pass
runs a second time, wider: every entry point must still return the bits of a default context."""
import numpy as np
import pytest

from oracle import tadpole_oracle as O
from tadpole_b200 import Context
from tadpole_b200.synth import synth_hic

pytestmark = pytest.mark.gpu
CAP = 8


def _narrow(devices=0):
    c = Context(devices)
    c.set("level_cap", CAP)
    return c


def _same(a, b):
    assert a["scores"].shape[1] > CAP                         # more levels than the first CH pass holds: the wide pass ran
    assert [a[key] for key in ("nf", "k", "n_pcs", "n_clusters")] == [b[key] for key in ("nf", "k", "n_pcs", "n_clusters")]
    assert np.array_equal(a["seqdist"], b["seqdist"]) and np.array_equal(a.get("bad"), b.get("bad"))
    assert a["scores"].shape == b["scores"].shape and np.array_equal(a["scores"], b["scores"], equal_nan=True)


def test_wide_sweep_equals_default_context(ctx):
    narrow = _narrow()
    m = synth_hic(400, seed=12)
    want = ctx.call(m)
    _same(narrow.call(m), want)
    keep = np.flatnonzero(~want["bad"]).astype(np.int32)
    _same(narrow.call_arm(keep), ctx.call_arm(keep))
    _same(narrow.recall(want["nf"], max_pcs=60, min_clusters=3), ctx.recall(want["nf"], max_pcs=60, min_clusters=3))
    (ncl_w, sc_w), (ncl, sc) = ctx.sweep(60), narrow.sweep(60)
    assert sc.shape == (60, ncl.max()) and sc.shape[1] > CAP
    assert np.array_equal(ncl, ncl_w) and np.array_equal(sc, sc_w, equal_nan=True)
    # a sweep that runs no candidate leaves no width or scores of the sweep before it
    ncl, sc = narrow.sweep(60, cand_begin=60)
    assert not ncl.any() and sc.shape == (60, 0) and narrow.dims()["maxlev"] == 0
    # the batch pool's contexts take the handle's level_cap
    mats = [m, synth_hic(300, seed=1), synth_hic(520, seed=2)]
    for mm, g in zip(mats, narrow.call_batch(mats, inflight=2, tables=False)):
        _same(g, ctx.call(mm))
    narrow.close()


@pytest.mark.parametrize("devices", [0, pytest.param([0, 1], marks=pytest.mark.skipif(
    "__import__('tadpole_b200')._lib.device_count() < 2", reason="needs >= 2 GPUs"))])
def test_wide_sweep_in_both_arms(ctx, devices):
    m = synth_hic(700, seed=5, centromere=True)
    lm = O.load_mat_numeric(m, centromere_search=True)
    kp, kq = np.asarray(lm.p.names) - 1, np.asarray(lm.q.names) - 1
    narrow = _narrow(devices)
    narrow.filter(m)
    got = narrow.call_arms(kp, kq)
    narrow.close()
    ctx.filter(m)
    for g, w in zip(got, ctx.call_arms(kp, kq)):
        _same(g, w)
