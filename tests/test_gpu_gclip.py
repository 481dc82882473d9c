"""Per-tensor gradient clipping on the GPU (lrcn_set_gclip / lrcn_grad_norms): every Adam path against the clip reference
(tests/gclip_ref.py: Knet's gclip! before the oracle's Adam) on the gradient the step actually used, the device norms against
fp64 norms of that gradient, gclip = 0 leaving the step exactly as it was, launch counts, graph replay with changing gclip,
trajectories, the workload sizes and the argument / state errors."""
import os

import numpy as np
import pytest
import torch

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, synth
from oracle import lrcn_oracle as O
import gclip_ref as R

pytestmark = pytest.mark.gpu

PRECS = [int(x) for x in os.environ.get("LRCN_TEST_PRECS", "0,1").split(",")]
RTOL = 1e-4
# the bars of test_adam_kernel_exact_on_given_gradient: (rtol, atol) for w, m, v
BARS = ((2e-6, 2e-8), (2e-6, 1e-12), (2e-6, 1e-14))


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))


def make(E, H1, H2, V, B, l, n_img=32, scale=3.0, seed=1):
    model = synth.initweights([H1, H2], V, E, seed=seed)
    model = [w * np.float32(scale) if w.shape[0] > 1 else w for w in model]
    feats = synth.features(n_img, seed=2) * np.float32(50)
    ids = np.arange(1, n_img + 1, dtype=np.int64)
    img = ids[synth.image_ids(B, n_img, seed=5) - 1]
    tok = synth.tokens(l, B, V, seed=3)
    return model, feats, ids, img, tok


def open_handle(E, H1, H2, V, B, l, prec, graphs=1):
    return abi.Handle(abi.default_config(embed=E, hidden1=H1, hidden2=H2, vocab=V, max_batch=B, max_len=max(l, 1), max_gen_rows=8,
                                         precision=prec, use_graphs=graphs))


def excess(got, want, rtol, atol):
    """max |got - want| in units of the bar atol + rtol |want| (<= 1: within the bar)"""
    want = np.asarray(want, np.float64)
    return float(np.max(np.abs(np.asarray(got, np.float64) - want) / (atol + rtol * np.abs(want))))


def set_random_adam_state(h, g_probe, rs, t=6):
    """Non-zero m, v sized like the gradient (at m = v = 0 an Adam step hardly depends on the gradient's scale)."""
    for k in range(1, 10):
        rms = float(np.sqrt(np.mean(np.square(g_probe[k - 1], dtype=np.float64)))) + 1e-12
        shape = g_probe[k - 1].shape
        h.set_adam_state(k, 0, (rs.standard_normal(shape) * 0.3 * rms).astype(np.float32))
        h.set_adam_state(k, 1, (rs.uniform(0.5, 1.5, shape) * rms * rms).astype(np.float32))
    h.set_adam_step(t)


def check_step_against_reference(h, step, gclip, rs, g_probe, min_each_side=3):
    """Check 1: give every tensor non-zero Adam state, read w, m, v, run `step`, read the gradient it used and apply the clip
    reference + the oracle's Adam to exactly those values.  Clipped tensors must match the clipped reference and be far from the
    unclipped one; the others must match the unclipped one.  Returns the number of clipped tensors."""
    set_random_adam_state(h, g_probe, rs)
    t0 = h.get_adam_step()
    w0 = h.get_model()
    m0 = [h.get_adam_state(k, 0) for k in range(1, 10)]
    v0 = [h.get_adam_state(k, 1) for k in range(1, 10)]
    h.set_gclip(gclip)
    step()
    assert h.get_adam_step() == t0 + 1
    g = [h.get_grad(k) for k in range(1, 10)]
    nrm = R.norms(g)
    clipped = (nrm > gclip) if gclip > 0 else np.zeros(9, bool)
    if gclip > 0:
        assert clipped.sum() >= min_each_side and (~clipped).sum() >= min_each_side, (gclip, nrm)
    refs = {}
    for name, c in (("clip", gclip), ("plain", 0.0)):
        w = [x.copy() for x in w0]
        opt = O.initparams(w)
        for p, m, v in zip(opt, m0, v0):
            p.fstm, p.scndm, p.t = m.copy(), v.copy(), t0
        R.update(w, g, opt, c)
        refs[name] = (w, [p.fstm for p in opt], [p.scndm for p in opt])
    for k in range(9):
        got = (h.get_param(k + 1), h.get_adam_state(k + 1, 0), h.get_adam_state(k + 1, 1))
        want = refs["clip"] if clipped[k] else refs["plain"]
        for i, (rt, at) in enumerate(BARS):
            assert excess(got[i], want[i][k], rt, at) <= 1.0, (k + 1, "wmv"[i], bool(clipped[k]), excess(got[i], want[i][k], rt, at))
        if clipped[k]:
            far = max(excess(got[i], refs["plain"][i][k], *BARS[i]) for i in range(2))
            assert far > 100, (k + 1, far)  # the clip has teeth: the unclipped update is far outside the bar
    return int(clipped.sum())


def probe_gradient(h, img, tok, pdrop=0.0, seed=0):
    h.grad(0, img, tok, pdrop, seed)
    return [h.get_grad(k) for k in range(1, 10)], h.grad_norms()


SMALL = dict(E=64, H1=64, H2=64, V=300, B=8, l=5)


def small_handle(prec, graphs=1):
    c = SMALL
    model, feats, ids, img, tok = make(c["E"], c["H1"], c["H2"], c["V"], c["B"], c["l"])
    h = open_handle(c["E"], c["H1"], c["H2"], c["V"], c["B"], c["l"], prec, graphs)
    h.set_model(model)
    h.load_features(0, ids, feats)
    return h, model, img, tok


# ----------------------------------------------------------------------------------------------------------------- 1
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("path", ["train_step", "grad_adam_update", "staged"])
def test_clip_exact_on_the_gradient_the_step_used(prec, path):
    """bf16x3 train_step / staged = the overlapped bucketed update (a norm launch before each bucket's Adam); fp32 train_step
    and lrcn_grad + lrcn_adam_update = the flat update (one whole-arena norm launch)."""
    rs = np.random.RandomState(7)
    h, model, img, tok = small_handle(prec)
    with h:
        g_probe, nrm = probe_gradient(h, img, tok, 0.4, 3)
        gclip = R.pick_gclip(nrm)
        h.stage_batch(0, 0, img, tok)
        steps = {"train_step": lambda: h.train_step(0, img, tok, 0.4, 3),
                 "grad_adam_update": lambda: (h.grad(0, img, tok, 0.4, 3), h.adam_update()),
                 "staged": lambda: (h.train_step_staged(0, 0.4, 3), h.sync())}
        for rep in range(2):  # the second step replays the captured graph
            check_step_against_reference(h, steps[path], gclip, rs, g_probe)


# ----------------------------------------------------------------------------------------------------------------- 2
@pytest.mark.parametrize("prec", PRECS)
def test_grad_norms_match_fp64_norms_and_are_reproducible(prec):
    h, model, img, tok = small_handle(prec)
    with h:
        with pytest.raises(abi.LrcnError) as ei:
            h.grad_norms()
        assert ei.value.code == abi.ERR_STATE
        h.loss(0, img, tok)  # a forward pass computes no gradient
        with pytest.raises(abi.LrcnError) as ei:
            h.grad_norms()
        assert ei.value.code == abi.ERR_STATE
        for step in (lambda: h.grad(0, img, tok, 0.4, 1), lambda: h.train_step(0, img, tok)):
            step()
            a = h.grad_norms()
            b = h.grad_norms()
            assert np.array_equal(a, b)
            want = R.norms([h.get_grad(k) for k in range(1, 10)])
            assert np.all(np.abs(a - want) <= 1e-12 * want), (a, want)
            assert np.all(a > 0)


# ----------------------------------------------------------------------------------------------------------------- 3
def test_gclip_off_is_bit_identical_to_never_setting_it():
    """fp32 mode, 3 train steps at pdrop 0.4: a handle that never calls the setter, one with gclip = 0 and one with gclip = 1e30
    (norm launches run, nothing clips) end with bit-identical w, m, v.  The shape keeps every fp32 reduction of the step
    independent of atomic order (no split-K GEMM with more than two slices over non-zero data, every token of the batch but bos
    distinct, features non-zero only in the first 64 dimensions), so the three runs can be compared bit for bit."""
    E = H = 32
    V, B, l = 200, 2, 5
    model = synth.initweights([H, H], V, E, seed=2)
    model = [w * np.float32(3) if w.shape[0] > 1 else w for w in model]
    feats = np.zeros((4, 4096), np.float32)
    feats[:, :64] = np.random.RandomState(3).uniform(0, 1, (4, 64))
    ids = np.arange(1, 5, dtype=np.int64)
    img = np.array([1, 3], dtype=np.int64)
    words = np.random.RandomState(4).permutation(np.arange(4, V + 1))[:3 * l * B].reshape(3, l, B).astype(np.int64)
    out = []
    for setting in (None, 0.0, 1e30):
        with open_handle(E, H, H, V, B, l, abi.PREC_FP32) as h:
            h.set_model(model)
            h.load_features(0, ids, feats)
            if setting is not None:
                h.set_gclip(setting)
            for s in range(3):
                h.train_step(0, img, words[s], 0.4, 100 + s)
            out.append([(h.get_param(k), h.get_adam_state(k, 0), h.get_adam_state(k, 1)) for k in range(1, 10)])
    for other in out[1:]:
        for k in range(9):
            for i in range(3):
                assert np.array_equal(out[0][k][i], other[k][i]), (k + 1, "wmv"[i])


# ----------------------------------------------------------------------------------------------------------------- 4
@pytest.mark.parametrize("prec", PRECS)
def test_launch_counts(prec):
    """gclip = 0 launches what a handle that never called the setter launches; gclip > 0 adds one norm launch per Adam launch:
    4 on the overlapped path (bf16x3 train step), 1 on the flat paths (fp32 train step, lrcn_adam_update)."""
    per_step = {}
    for setting in (None, 0.0, 1e30):
        h, model, img, tok = small_handle(prec)
        with h:
            if setting is not None:
                h.set_gclip(setting)
            h.train_step(0, img, tok)  # capture
            n0 = h.kernel_launches()
            h.train_step(0, img, tok)
            n1 = h.kernel_launches()
            h.grad(0, img, tok)
            n2 = h.kernel_launches()
            h.adam_update()
            n3 = h.kernel_launches()
            per_step[setting] = (n1 - n0, n3 - n2)
    assert per_step[0.0] == per_step[None]
    extra = 4 if prec == abi.PREC_BF16X3 else 1
    assert per_step[1e30] == (per_step[None][0] + extra, per_step[None][1] + 1), per_step


# ----------------------------------------------------------------------------------------------------------------- 5
@pytest.mark.parametrize("prec", PRECS)
def test_graph_replay_picks_up_every_gclip(prec):
    """With graphs on, steps at gclip = a, b, 0, a: a value baked into a captured graph would fail the check."""
    rs = np.random.RandomState(11)
    h, model, img, tok = small_handle(prec, graphs=1)
    with h:
        g_probe, nrm = probe_gradient(h, img, tok)
        a = R.pick_gclip(nrm)
        b = R.pick_gclip(nrm, avoid=a)
        counts = [check_step_against_reference(h, lambda: h.train_step(0, img, tok), g, rs, g_probe) for g in (a, b, 0.0, a)]
        assert counts[0] == counts[3] and counts[0] != counts[1] and counts[2] == 0


# ----------------------------------------------------------------------------------------------------------------- 6
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("pdrop", [0.0, 0.4])
def test_clipped_train_steps_match_oracle_trajectory(prec, pdrop):
    """Three clipped train steps against the oracle's (clip reference + Adam) trajectory at the bars of
    test_train_steps_match_oracle_adam.  gclip is re-chosen before every step from the oracle's gradient norms."""
    c = SMALL
    E, H1, H2, V, B, l = c["E"], c["H1"], c["H2"], c["V"], c["B"], c["l"]
    model, feats, ids, img, tok = make(E, H1, H2, V, B, l)
    X = feats[img - 1]
    ref = [w.copy() for w in model]
    opt = O.initparams(ref)
    with open_handle(E, H1, H2, V, B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        n_clipped = 0
        for step in range(3):
            seed = 50 + step
            masks = O.dropout_masks(pdrop, seed, l + 1, B, E, H2) if pdrop > 0 else None
            g_ref, L_ref = O.lossgradient(ref, O.initstate(ref, B), X, list(tok), range(0, l), masks=masks)
            gclip = R.pick_gclip(R.norms(g_ref))
            n_clipped += int((R.norms(g_ref) > gclip).sum())
            R.update(ref, g_ref, opt, gclip)
            h.set_gclip(gclip)
            L = h.train_step(0, img, tok, pdrop, seed)
            assert abs(L - L_ref) < RTOL * abs(L_ref), f"step {step}"
        assert n_clipped >= 9 and h.get_adam_step() == 3
        for k in range(1, 10):
            d_ref = ref[k - 1] - model[k - 1]
            assert relerr(h.get_param(k) - model[k - 1], d_ref) < 5e-3, f"param {k}"
            assert relerr(h.get_adam_state(k, 0), opt[k - 1].fstm) < 2e-4, f"m of param {k}"
            assert relerr(h.get_adam_state(k, 1), opt[k - 1].scndm) < 4e-4, f"v of param {k}"


@pytest.mark.parametrize("prec", PRECS)
def test_clipped_train_epoch_equals_per_step_calls(prec):
    """lrcn_train_epoch under clipping == the same batches through lrcn_train_step, at the epoch test's tolerance."""
    E, H1, H2, V, B = 64, 64, 64, 300, 8
    model, feats, ids, _, _ = make(E, H1, H2, V, B, 5)
    blens = [5, 3, 7, 4]
    seq = np.concatenate([synth.tokens(l, B, V, seed=70 + b) for b, l in enumerate(blens)])
    img = np.stack([ids[synth.image_ids(B, len(ids), seed=80 + b) - 1] for b in range(len(blens))])
    order = np.array([2, 0, 3, 1], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(blens)])
    with open_handle(E, H1, H2, V, B, 8, prec) as h, open_handle(E, H1, H2, V, B, 8, prec) as h2:
        for x in (h, h2):
            x.set_model(model)
            x.load_features(0, ids, feats)
        _, nrm = probe_gradient(h2, img[2], seq[starts[2]:starts[2] + blens[2]], 0.4, 11)
        gclip = R.pick_gclip(nrm)
        for x in (h, h2):
            x.set_gclip(gclip)
        losses = h.train_epoch(0, seq, img, blens, order, 0.4, seed=11)
        want = []
        for n, b in enumerate(order):
            want.append(h2.train_step(0, img[b], seq[starts[b]:starts[b] + blens[b]], 0.4, 11 + n))
            if n == 0:
                assert (h2.grad_norms() > gclip).sum() >= 3  # the epoch really clips
        assert h.get_adam_step() == h2.get_adam_step() == 4
        np.testing.assert_allclose(losses, want, rtol=1e-6)
        for k in range(1, 10):
            assert relerr(h.get_param(k) - model[k - 1], h2.get_param(k) - model[k - 1]) < 1e-3, f"param {k}"
            assert relerr(h.get_adam_state(k, 0), h2.get_adam_state(k, 0)) < 1e-3, f"adam m {k}"


# ----------------------------------------------------------------------------------------------------------------- 7
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("shape", ["flickr30k_train_b256", "coco_2f"])
def test_clip_exact_at_workload_sizes(prec, shape):
    E, H, V, B, l = {"flickr30k_train_b256": (512, 512, 7731, 256, 16), "coco_2f": (1000, 1000, 10636, 256, 12)}[shape]
    rs = np.random.RandomState(13)
    model = synth.initweights([H, H], V, E, seed=1)
    model = [w * np.float32(1.5) if w.shape[0] > 1 else w for w in model]
    feats = synth.features(128, seed=2) * np.float32(50)
    ids = np.arange(1, 129, dtype=np.int64)
    img = synth.image_ids(B, 128, seed=5)
    tok = synth.tokens(l, B, V, seed=3, zipf=True)
    with open_handle(E, H, H, V, B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        g_probe, nrm = probe_gradient(h, img, tok, 0.4, 9)
        check_step_against_reference(h, lambda: h.train_step(0, img, tok, 0.4, 9), R.pick_gclip(nrm), rs, g_probe)


# ----------------------------------------------------------------------------------------------------------------- 8
def test_bad_gclip_is_refused_and_the_previous_value_stays():
    h, model, img, tok = small_handle(abi.PREC_FP32)
    with h:
        h.set_gclip(1e30)
        h.train_step(0, img, tok)
        n0 = h.kernel_launches()
        h.train_step(0, img, tok)
        per_step = h.kernel_launches() - n0
        for bad in (-1.0, float("nan"), float("inf"), -float("inf")):
            with pytest.raises(abi.LrcnError) as ei:
                h.set_gclip(bad)
            assert ei.value.code == abi.ERR_ARG
        n0 = h.kernel_launches()
        h.train_step(0, img, tok)
        assert h.kernel_launches() - n0 == per_step  # still clipping (the norm launch is still there)
        h.set_gclip(0.0)
        n0 = h.kernel_launches()
        h.train_step(0, img, tok)
        assert h.kernel_launches() - n0 == per_step - 1


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="a group handle needs two GPUs")
def test_group_handle_refuses_clipping():
    cfg = abi.default_config(embed=64, hidden1=64, hidden2=64, vocab=300, max_batch=8, max_len=5, max_gen_rows=8, n_gpus=2)
    with abi.Handle(cfg) as h:
        h.set_gclip(0.0)  # off is always fine
        for call in (lambda: h.set_gclip(1.0), h.grad_norms):
            with pytest.raises(abi.LrcnError) as ei:
                call()
            assert ei.value.code == abi.ERR_STATE
