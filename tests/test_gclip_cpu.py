"""Per-tensor gradient clipping (Knet Adam(gclip=...)) without a GPU: the clip reference the GPU tests compare against, and the
host mirror's gclip option reaching the library."""
import numpy as np
import pytest

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, host, synth
from oracle import lrcn_oracle as O
import gclip_ref as R


def case(seed=0):
    model = synth.initweights([16, 24], 37, 8, seed=seed + 1)
    rs = np.random.RandomState(seed)
    # gradients of very different sizes, like the nine real ones; one all-zero tensor
    g = [(rs.standard_normal(w.shape) * 10.0 ** rs.uniform(-4, 1)).astype(np.float32) for w in model]
    g[4][:] = 0
    return model, g


def run(model, g, gclip=None, steps=2):
    w = [x.copy() for x in model]
    opt = O.initparams(w)
    for _ in range(steps):
        if gclip is None:
            O.update(w, g, opt)
        else:
            R.update(w, g, opt, gclip)
    return w, opt


@pytest.mark.parametrize("gclip", [0.0, "max", 1e30])
def test_off_or_above_every_norm_is_bit_identical_to_no_clipping(gclip):
    model, g = case()
    if gclip == "max":
        gclip = float(R.norms(g).max())  # a norm equal to gclip is not clipped (clip when |g| > gclip)
    w0, opt0 = run(model, g)
    w1, opt1 = run(model, g, gclip)
    for a, b, p, q in zip(w0, w1, opt0, opt1):
        assert np.array_equal(a, b) and np.array_equal(p.fstm, q.fstm) and np.array_equal(p.scndm, q.scndm)


def test_clipped_tensor_has_norm_gclip_same_direction_and_others_unchanged():
    model, g = case(3)
    before = [x.copy() for x in g]
    nrm = R.norms(g)
    gclip = R.pick_gclip(nrm)
    out = R.clip(g, gclip)
    assert all(np.array_equal(a, b) for a, b in zip(g, before)), "the caller's gradient must not be modified"
    clipped = nrm > gclip
    assert 3 <= clipped.sum() <= 6
    for k in range(9):
        if clipped[k]:
            n = np.linalg.norm(out[k].astype(np.float64))
            assert abs(n - gclip) <= 1e-6 * gclip
            cos = np.vdot(out[k].astype(np.float64), g[k].astype(np.float64)) / (n * nrm[k])
            assert cos > 1 - 1e-12
        else:
            assert out[k] is g[k]
    assert out[4] is g[4]  # a zero tensor is never scaled
    # only the clipped tensors' Adam update changes
    w0, _ = run(model, g, 0.0, steps=1)
    w1, _ = run(model, g, gclip, steps=1)
    for k in range(9):
        assert np.array_equal(w0[k], w1[k]) != bool(clipped[k]), k


def test_pick_gclip_leaves_three_on_each_side():
    rs = np.random.RandomState(5)
    for _ in range(50):
        nrm = 10.0 ** rs.uniform(-5, 3, 9)
        t = R.pick_gclip(nrm)
        assert 3 <= (nrm > t).sum() <= 6
        t2 = R.pick_gclip(nrm, avoid=t)
        assert 3 <= (nrm > t2).sum() <= 6 and (nrm > t2).sum() != (nrm > t).sum()


class RecordingHandle:
    def __init__(self, cfg):
        self.cfg = cfg
        self.calls = []

    def set_gclip(self, g):
        self.calls.append(("set_gclip", g))

    def close(self):
        pass


def test_host_lrcn_gclip_reaches_set_gclip(monkeypatch):
    monkeypatch.setattr(abi, "Handle", RecordingHandle)
    assert host.LRCN([8, 8], 20, 8, 2).h.calls == []  # the default is the reference: the setter is never called
    assert host.LRCN([8, 8], 20, 8, 2, gclip=0.0).h.calls == []
    assert host.LRCN([8, 8], 20, 8, 2, gclip=2.5).h.calls == [("set_gclip", 2.5)]
