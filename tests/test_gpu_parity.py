"""GPU parity tests: the CUDA path, called through the C ABI (ctypes), against the CPU oracle on the
same seeded inputs.  Bars (BASELINE.json north_star): integer/index work bit-exact; loss and the nine
gradients within 1e-4 relative; >=99% identical captions, token log-probs within 1e-4."""
import numpy as np
import pytest

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, host, synth
from oracle import lrcn_oracle as O

pytestmark = pytest.mark.gpu

import os

PRECS = [int(x) for x in os.environ.get("LRCN_TEST_PRECS", "0,1").split(",")]  # 0 = fp32 CUDA cores, 1 = bf16x3 tcgen05
RTOL = 1e-4  # north_star: "per-step loss and gradients agree within 1e-4 relative in fp32"


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))


def make_case(E, H1, H2, V, B, l, n_img=32, scale=3.0, fscale=50.0, seed=1, zipf=False):
    model = synth.initweights([H1, H2], V, E, seed=seed)
    model = [w * np.float32(scale) if w.shape[0] > 1 else w for w in model]
    feats = synth.features(n_img, seed=2) * np.float32(fscale)
    ids = np.arange(1, n_img + 1, dtype=np.int64) * 7 + 100  # non-trivial image ids
    img = ids[synth.image_ids(B, n_img, seed=5) - 1]
    tok = synth.tokens(l, B, V, seed=3, zipf=zipf)
    X = feats[(img - 100) // 7 - 1]
    return model, feats, ids, img, tok, X


def open_handle(E, H1, H2, V, B, l, prec, gen_rows=64, graphs=1, hooks=False):
    cfg = abi.default_config(embed=E, hidden1=H1, hidden2=H2, vocab=V, max_batch=B, max_len=max(l, 1), max_gen_rows=gen_rows,
                             precision=prec, use_graphs=graphs)
    return abi.Handle(cfg, hooks=hooks)  # hooks=True: liblrcn_b200_test.so (product objects + kernel-level test hooks)


# ----------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("aK,bK", [(1, 1), (1, 0), (0, 0), (0, 1)])
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (200, 136, 520), (64, 2048, 512), (777, 1000, 333)])
def test_gemm_kernels(prec, aK, bK, M, N, K):
    rs = np.random.RandomState(M + N + K)
    A = rs.standard_normal((M, K)).astype(np.float32)
    B = rs.standard_normal((K, N)).astype(np.float32)
    bias = rs.standard_normal(N).astype(np.float32)
    C0 = rs.standard_normal((M, N)).astype(np.float32)
    ref = A.astype(np.float64) @ B.astype(np.float64)
    with open_handle(64, 64, 64, 100, 4, 2, prec, 4, hooks=True) as h:
        out = h.test_gemm(prec, aK, bK, A if aK else np.ascontiguousarray(A.T), np.ascontiguousarray(B.T) if bK else B)
        assert relerr(out, ref) < 2e-5
        out = h.test_gemm(prec, aK, bK, A if aK else np.ascontiguousarray(A.T), np.ascontiguousarray(B.T) if bK else B, bias, C0)
        assert relerr(out, ref + bias + C0) < 2e-5


@pytest.mark.parametrize("aK,bK", [(1, 1), (1, 0), (0, 0), (0, 1)])
@pytest.mark.parametrize("M,N,K", [(1344, 2056, 512),   # CTA-pair kernel, whole 256x256 tiles, ragged N (TMA store clips)
                                   (1000, 500, 3840),   # CTA-pair kernel, stream-K: partial tiles summed by TMA reduce-add
                                   (1536, 520, 4100)])  # stream-K with ragged N and K
def test_gemm_pair_kernel_and_streamk(aK, bK, M, N, K):
    if 1 not in PRECS:
        pytest.skip("bf16x3 precision not selected")
    rs = np.random.RandomState(M + N + K)
    A = rs.standard_normal((M, K)).astype(np.float32)
    B = rs.standard_normal((K, N)).astype(np.float32)
    bias = rs.standard_normal(N).astype(np.float32)
    C0 = rs.standard_normal((M, N)).astype(np.float32)
    ref = A.astype(np.float64) @ B.astype(np.float64)
    Ain = A if aK else np.ascontiguousarray(A.T)
    Bin = np.ascontiguousarray(B.T) if bK else B
    with open_handle(64, 64, 64, 100, 4, 2, 1, 4, hooks=True) as h:
        assert relerr(h.test_gemm(1, aK, bK, Ain, Bin), ref) < 2e-5
        assert relerr(h.test_gemm(1, aK, bK, Ain, Bin, bias, None), ref + bias) < 2e-5
        assert relerr(h.test_gemm(1, aK, bK, Ain, Bin, bias, C0), ref + bias + C0) < 2e-5


@pytest.mark.parametrize("prec", PRECS)
def test_param_roundtrip_bit_exact(prec):
    E, H1, H2, V = 24, 16, 32, 57
    model = synth.initweights([H1, H2], V, E, seed=3)
    with open_handle(E, H1, H2, V, 4, 3, prec) as h:
        for k in range(1, 10):
            assert h.param_shape(k) == model[k - 1].shape
        h.set_model(model)
        back = h.get_model()
        for a, b in zip(model, back):
            assert a.shape == b.shape and np.array_equal(a, b)
        with pytest.raises(abi.LrcnError) as ei:
            h.set_param(1, np.zeros((3, 3), np.float32))
        assert ei.value.code == abi.ERR_ARG


def test_beam_selection_bit_exact_given_identical_probs():
    # "embedding indices and the beam-search integer selection are bit-exact given identical logits"
    rs = np.random.RandomState(5)
    n_img, K, V = 7, 3, 1000
    for first in (1, 0):
        probs = rs.dirichlet(np.ones(V) * 0.05, size=n_img * K).astype(np.float32)
        probs[0, 10] = probs[0, 400] = probs[0].max() + np.float32(0.1)      # exact ties inside a row
        probs[4] = probs[3]                                                  # exact ties across beams
        parent = rs.uniform(0.1, 1, n_img * K).astype(np.float32)
        parent[4] = parent[3]
        with open_handle(64, 64, 64, 100, 4, 2, abi.PREC_FP32, hooks=True) as h:
            tok, par, sc = h.test_beam_select(probs, parent, n_img, K, first)
        for img in range(n_img):
            cands = []
            for b in range(1 if first else K):
                r = img * K + b
                top = np.argsort(-probs[r], kind="stable")[:K]  # ties -> lower index (lrcn.jl:655)
                for j in top:
                    cands.append((int(j) + 1, np.float32(probs[r, j] * parent[r]), b))
            order = np.argsort(-np.array([c[1] for c in cands], np.float32), kind="stable")[:K]  # lrcn.jl:667
            assert tok[img].tolist() == [cands[o][0] for o in order]
            assert par[img].tolist() == [cands[o][2] for o in order]
            assert np.array_equal(sc[img], np.array([cands[o][1] for o in order], np.float32))


# ----------------------------------------------------------------------------- loss / gradient
CASES = [
    dict(E=8, H1=8, H2=16, V=23, B=3, l=4),        # tiny, ragged tiles everywhere
    dict(E=64, H1=64, H2=64, V=300, B=8, l=5),
    dict(E=128, H1=192, H2=128, V=1111, B=24, l=11, zipf=True),
    dict(E=40, H1=24, H2=72, V=131, B=5, l=3),      # C = 36 is not a multiple of 8 -> padded ld of v/dv (the coco_2f C=500 case)
    dict(E=64, H1=512, H2=512, V=300, B=80, l=7, scale=1.5),   # bench-sized hidden state: 8 k-blocks, 2 m-tiles (second one ragged)
    dict(E=64, H1=640, H2=320, V=200, B=70, l=4, scale=1.5),   # H1 too large for weight residency -> per-step kernels for layer 1
    dict(E=104, H1=200, H2=200, V=333, B=33, l=5, scale=2.0),  # coco_2f-like ragged dims (H=1000 there): K, N not multiples of 64/16
    dict(E=64, H1=64, H2=64, V=300, B=2048, l=3),   # the largest batch the persistent LSTM kernels take (32 m-tiles x 2 chains)
    dict(E=64, H1=64, H2=64, V=300, B=2049, l=3),   # one row more: per-step LSTM kernels
]


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", CASES)
@pytest.mark.parametrize("graphs", [0, 1])
def test_loss_and_gradients_match_oracle(prec, case, graphs, monkeypatch):
    if graphs == 0 and prec == abi.PREC_BF16X3:
        monkeypatch.setenv("LRCN_NO_PERSISTENT", "1")  # graphs=0 runs double as the per-step LSTM kernel coverage
    c = dict(case)
    zipf = c.pop("zipf", False)
    model, feats, ids, img, tok, X = make_case(**c, zipf=zipf)
    B, l = c["B"], c["l"]
    g_ref, L_ref = O.lossgradient(model, O.initstate(model, B), X, list(tok), range(0, l))
    lp_ref = O.token_logps(model, O.initstate(model, B), X, list(tok), range(0, l))
    with open_handle(c["E"], c["H1"], c["H2"], c["V"], B, l, prec, graphs=graphs) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        s, n = h.loss(0, img, tok)
        assert n == B * (l + 1)
        assert abs(-s / n - L_ref) < RTOL * abs(L_ref)
        np.testing.assert_allclose(h.token_logps(l, B), lp_ref, rtol=RTOL, atol=1e-5)
        for rep in range(2):  # second call replays the cached CUDA graph
            L = h.grad(0, img, tok)
            assert abs(L - L_ref) < RTOL * abs(L_ref)
            for k in range(1, 10):
                assert relerr(h.get_grad(k), g_ref[k - 1]) < RTOL, f"gradient of param {k} (rep {rep})"
        # embedding gradient: rows of unused words are exactly zero; bos row accumulates B contributions
        gW = h.get_grad(7)
        used = {O.BOS - 1} | {int(t) - 1 for t in tok.ravel()}
        unused = sorted(set(range(c["V"])) - used)
        assert np.abs(gW[unused]).sum() == 0
        assert np.abs(gW[O.BOS - 1]).sum() > 0


@pytest.mark.parametrize("prec", PRECS)
def test_untrained_loss_is_ln_vocab(prec):
    # known answer from the reference's slides: epoch-0 loss = ln V (8.953 Flickr30k, 9.272 COCO)
    V = 7731
    E, H1, H2, B, l = 64, 64, 64, 16, 6
    model, feats, ids, img, tok, X = make_case(E, H1, H2, V, B, l)
    model[7][:] = 0
    model[8][:] = 0
    with open_handle(E, H1, H2, V, B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        s, n = h.loss(0, img, tok)
        assert abs(-s / n - np.log(V)) < 1e-5 * np.log(V)
        assert round(-s / n, 3) == 8.953


@pytest.mark.parametrize("prec", PRECS)
def test_train_steps_match_oracle_adam(prec):
    E, H1, H2, V, B, l = 64, 64, 64, 300, 8, 5
    model, feats, ids, img, tok, X = make_case(E, H1, H2, V, B, l)
    ref = [w.copy() for w in model]
    opt = O.initparams(ref)
    with open_handle(E, H1, H2, V, B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        for step in range(3):
            L_ref = O.train_step(ref, opt, X, list(tok), range(0, l))
            L = h.train_step(0, img, tok)
            assert abs(L - L_ref) < RTOL * abs(L_ref), f"step {step}"
        assert h.get_adam_step() == 3
        for k in range(1, 10):
            # Adam's first steps move every weight by ~lr regardless of |g|: compare the UPDATE, not the weight
            d_ref = ref[k - 1] - model[k - 1]
            d = h.get_param(k) - model[k - 1]
            assert relerr(d, d_ref) < 5e-3, f"param {k}"
            assert relerr(h.get_adam_state(k, 0), opt[k - 1].fstm) < 2e-4, f"m of param {k}"
            assert relerr(h.get_adam_state(k, 1), opt[k - 1].scndm) < 4e-4, f"v of param {k}"


def test_adam_kernel_exact_on_given_gradient():
    # Adam alone on a known gradient/moment state: same op order as the oracle -> tight tolerance
    E, H1, H2, V = 16, 16, 16, 40
    model = synth.initweights([H1, H2], V, E, seed=4)
    rs = np.random.RandomState(1)
    with open_handle(E, H1, H2, V, 4, 3, abi.PREC_FP32) as h:
        h.set_model(model)
        ref = [w.copy() for w in model]
        opt = O.initparams(ref)
        for p, w in zip(opt, ref):
            p.fstm = (rs.standard_normal(w.shape) * 1e-3).astype(np.float32)
            p.scndm = (rs.uniform(0, 1e-5, w.shape)).astype(np.float32)
            p.t = 6
        for k in range(1, 10):
            h.set_adam_state(k, 0, opt[k - 1].fstm)
            h.set_adam_state(k, 1, opt[k - 1].scndm)
        h.set_adam_step(6)
        # run a grad to have gradients on device, then fetch them and apply the oracle's Adam to the same values
        feats = synth.features(8) * np.float32(50)
        ids = np.arange(1, 9, dtype=np.int64)
        h.load_features(0, ids, feats)
        tok = synth.tokens(3, 4, V)
        h.grad(0, ids[:4], tok)
        g = [h.get_grad(k) for k in range(1, 10)]
        O.update(ref, g, opt)
        h.adam_update()
        assert h.get_adam_step() == 7
        for k in range(1, 10):
            np.testing.assert_allclose(h.get_param(k), ref[k - 1], rtol=2e-6, atol=2e-8)
            np.testing.assert_allclose(h.get_adam_state(k, 0), opt[k - 1].fstm, rtol=2e-6, atol=1e-12)
            np.testing.assert_allclose(h.get_adam_state(k, 1), opt[k - 1].scndm, rtol=2e-6, atol=1e-14)


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("case", [dict(E=64, H1=64, H2=64, V=300, B=16, l=5), dict(E=128, H1=192, H2=128, V=1111, B=24, l=11, zipf=True),
                                  dict(E=64, H1=512, H2=512, V=300, B=80, l=7, scale=1.5)])
def test_dropout_matches_oracle_with_the_same_masks(prec, case):
    """The reference trains at pdrop = 0.4 only (lrcn.jl:227; sites lrcn.jl:542,547).  Knet's RNG is not reproducible, so the
    oracle is handed the masks the CUDA path draws (its counter hash restated in oracle.dropout_masks): loss and the nine
    gradients must agree to 1e-4 like at p = 0; plus seed determinism, the Bernoulli keep rate and the 1/(1-p) scale."""
    c = dict(case)
    zipf = c.pop("zipf", False)
    model, feats, ids, img, tok, X = make_case(**c, zipf=zipf)
    E, H2, B, l = c["E"], c["H2"], c["B"], c["l"]
    T, p, seed = l + 1, 0.4, 20240611
    masks = O.dropout_masks(p, seed, T, B, E, H2)
    for M in masks:  # empirical keep rate (Bernoulli(1-p) within 4 sigma) and Knet's survivor scale 1/(1-p)
        assert abs(float((M > 0).mean()) - (1 - p)) < 4 * np.sqrt(p * (1 - p) / M.size)
        assert np.unique(M).tolist() == [0.0, float(np.float32(1) / (np.float32(1) - np.float32(p)))]
    g_ref, L_ref = O.lossgradient(model, O.initstate(model, B), X, list(tok), range(0, l), masks=masks)
    g0_ref, L0_ref = O.lossgradient(model, O.initstate(model, B), X, list(tok), range(0, l))
    assert abs(L_ref - L0_ref) > 1e-6 * abs(L0_ref)  # the masks do change the loss
    with open_handle(c["E"], c["H1"], c["H2"], c["V"], B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        for rep in range(2):  # second call replays the CUDA graph: the seed travels in the step scalars, not in the graph
            L = h.grad(0, img, tok, p, seed)
            assert abs(L - L_ref) < RTOL * abs(L_ref), (L, L_ref, L0_ref)
            for k in range(1, 10):
                assert relerr(h.get_grad(k), g_ref[k - 1]) < RTOL, f"gradient of param {k} at pdrop {p} (rep {rep})"
        other = h.grad(0, img, tok, p, seed + 1)
        assert abs(other - L) > 1e-6 * abs(L)          # another seed draws other masks
        assert abs(h.grad(0, img, tok, 0.0, seed) - L0_ref) < RTOL * abs(L0_ref)  # p = 0 is the identity
        # a train step at p = 0.4 is the oracle's Adam step on the masked gradient
        ref = [w.copy() for w in model]
        O.update(ref, g_ref, O.initparams(ref))
        Lt = h.train_step(0, img, tok, p, seed)
        assert abs(Lt - L_ref) < RTOL * abs(L_ref)
        for k in (1, 3, 7, 8):
            d_ref = ref[k - 1] - model[k - 1]
            assert relerr(h.get_param(k) - model[k - 1], d_ref) < 5e-3, f"Adam update of param {k}"
        with pytest.raises(abi.LrcnError):
            h.grad(0, img, tok, 1.0, 1)


@pytest.mark.parametrize("prec", PRECS)
def test_small_batch_then_large_batch_on_one_handle(prec):
    """average_loss runs B = 10 (lrcn.jl:260-269) on the handle that trains at a larger batch: slot t of the small call lands
    inside slot 0 (= h_0 = c_0 = 0, lrcn.jl:512-526) of the next larger one, which must therefore be re-zeroed every step."""
    E, H1, H2, V, l = 64, 128, 128, 300, 6
    model, feats, ids, img, tok, X = make_case(E, H1, H2, V, 48, l)
    for graphs in (1, 0):
        with open_handle(E, H1, H2, V, 48, l, prec, graphs=graphs) as h:
            h.set_model(model)
            h.load_features(0, ids, feats)
            for B in (10, 48, 7, 48):
                g_ref, L_ref = O.lossgradient(model, O.initstate(model, B), X[:B], list(tok[:, :B]), range(0, l))
                s, n = h.loss(0, img[:B], np.ascontiguousarray(tok[:, :B]))
                assert abs(-s / n - L_ref) < RTOL * abs(L_ref), (B, graphs)
                L = h.grad(0, img[:B], np.ascontiguousarray(tok[:, :B]))
                assert abs(L - L_ref) < RTOL * abs(L_ref), (B, graphs)
                for k in range(1, 10):
                    assert relerr(h.get_grad(k), g_ref[k - 1]) < RTOL, f"B={B} graphs={graphs} param {k}"


@pytest.mark.parametrize("prec", PRECS)
def test_staged_train_steps_match_host_buffer_steps_and_oracle(prec):
    """lrcn_train_step_staged (the call bench.py's `value` is timed on) == lrcn_train_step == the oracle, including
    back-to-back un-synchronised calls on slots of different lengths (the step scalars travel through a pinned ring)."""
    E, H1, H2, V, B = 64, 64, 64, 300, 8
    model, feats, ids, _, _, _ = make_case(E, H1, H2, V, B, 5)
    batches = []
    for s_, l in enumerate((5, 3, 7, 5)):
        img = ids[synth.image_ids(B, len(ids), seed=50 + s_) - 1]
        batches.append((img, synth.tokens(l, B, V, seed=60 + s_), l))
    ref = [w.copy() for w in model]
    opt = O.initparams(ref)
    with open_handle(E, H1, H2, V, B, 8, prec) as h, open_handle(E, H1, H2, V, B, 8, prec) as h2:
        for x in (h, h2):
            x.set_model(model)
            x.load_features(0, ids, feats)
        for s_, (img, tok, l) in enumerate(batches):
            h.stage_batch(s_, 0, img, tok)
        losses = []
        for rep in range(2):
            for s_, (img, tok, l) in enumerate(batches):
                Xb = feats[(img - 100) // 7 - 1]
                L_ref = O.train_step(ref, opt, Xb, list(tok), range(0, l))
                if rep == 0:
                    L = h.train_step_staged(s_, 0.0, 0, want_loss=True)
                    assert abs(L - L_ref) < RTOL * abs(L_ref), (s_, L, L_ref)
                else:
                    h.train_step_staged(s_, 0.0, 0)  # no D2H, no synchronisation between the four steps
                L2 = h2.train_step(0, img, tok)
                losses.append((L_ref, L2))
                assert abs(L2 - L_ref) < 2 * RTOL * abs(L_ref)
        h.sync()
        assert h.get_adam_step() == h2.get_adam_step() == 8
        for k in range(1, 10):
            a, b = h.get_param(k), h2.get_param(k)
            assert relerr(a - model[k - 1], b - model[k - 1]) < 1e-3, f"staged vs host-buffer steps, param {k}"
            assert relerr(a - model[k - 1], ref[k - 1] - model[k - 1]) < 2e-2, f"staged steps vs oracle, param {k}"


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("pdrop", [0.0, 0.4])
def test_train_epoch_on_device_equals_per_step_calls_and_oracle(prec, pdrop):
    """lrcn_train_epoch (SURVEY 8 row f-1: the epoch's batches are staged by a device kernel from resident data, image ids are
    resolved on the device, no per-step host work) == the same batches through lrcn_train_step, step for step: same losses,
    same weights, same Adam state -- and == the oracle's epoch at pdrop 0.  Covers the shuffled order, a batch that is
    skipped because l > max_len (lrcn.jl:353), a repeated batch, an l = 1 batch and non-contiguous image ids."""
    E, H1, H2, V, B = 64, 64, 64, 300, 8
    model, feats, ids, _, _, _ = make_case(E, H1, H2, V, B, 5)
    blens = [5, 3, 9, 1, 7, 8]          # 9 > max_len = 8: skipped
    seq = np.concatenate([synth.tokens(l, B, V, seed=70 + b) for b, l in enumerate(blens)])          # [sum l][B], 1-based
    img = np.stack([ids[synth.image_ids(B, len(ids), seed=80 + b) - 1] for b in range(len(blens))])   # [n_batches][B]
    order = np.array([4, 0, 2, 5, 3, 1, 0], dtype=np.int64)
    starts = np.concatenate([[0], np.cumsum(blens)])
    with open_handle(E, H1, H2, V, B, 8, prec) as h, open_handle(E, H1, H2, V, B, 8, prec) as h2:
        for x in (h, h2):
            x.set_model(model)
            x.load_features(0, ids, feats)
        losses = h.train_epoch(0, seq, img, blens, order, pdrop, seed=11)
        ref = [w.copy() for w in model]
        opt = O.initparams(ref)
        want, n = [], 0
        for b in order:
            l = blens[b]
            if l > 8:
                continue
            tok = seq[starts[b]:starts[b] + l]
            want.append(h2.train_step(0, img[b], tok, pdrop, 11 + n))
            n += 1
            if pdrop == 0.0:
                L_ref = O.train_step(ref, opt, feats[(img[b] - 100) // 7 - 1], list(tok), range(0, l))
                assert abs(want[-1] - L_ref) < 2 * RTOL * abs(L_ref)
        assert len(losses) == 6 and h.get_adam_step() == h2.get_adam_step() == 6
        # the same kernels on the same staged integers; fp32 atomics (loss sum, embedding gradient) reorder between runs
        np.testing.assert_allclose(losses, want, rtol=1e-6)
        for k in range(1, 10):
            assert relerr(h.get_param(k) - model[k - 1], h2.get_param(k) - model[k - 1]) < 1e-3, f"param {k}"
            assert relerr(h.get_adam_state(k, 0), h2.get_adam_state(k, 0)) < 1e-3, f"adam m {k}"
            if pdrop == 0.0:
                assert relerr(h.get_param(k) - model[k - 1], ref[k - 1] - model[k - 1]) < 2e-2, f"epoch vs oracle, param {k}"
        # forward-only epoch (average_loss, lrcn.jl:407-486) == the per-batch lrcn_loss calls
        s_e, n_e = h.loss_epoch(0, seq, img, blens)
        per = [h2.loss(0, img[b], seq[starts[b]:starts[b] + blens[b]]) for b in range(len(blens)) if blens[b] <= 8]
        assert n_e == sum(p_[1] for p_ in per) == B * sum(l + 1 for l in blens if l <= 8)
        assert abs(s_e - sum(p_[0] for p_ in per)) < 1e-5 * abs(s_e)
        # natural order (order = None) and a second epoch on the same handle (buffers are reused)
        l2 = h.train_epoch(0, seq, img, blens, None, pdrop, seed=30)
        w2 = [h2.train_step(0, img[b], seq[starts[b]:starts[b] + blens[b]], pdrop, 30 + i)
              for i, b in enumerate(b for b in range(len(blens)) if blens[b] <= 8)]
        np.testing.assert_allclose(l2, w2, rtol=1e-5)
        # an image id without features fails the call before any step runs; a token outside the vocabulary is reported
        before = h.get_param(9).copy()
        bad = img.copy()
        bad[3, 2] = 999999
        with pytest.raises(abi.LrcnError) as ei:
            h.train_epoch(0, seq, bad, blens, order, pdrop, seed=1)
        assert ei.value.code == abi.ERR_MISSING
        assert np.array_equal(h.get_param(9), before) and h.get_adam_step() == 11
        badseq = seq.copy()
        badseq[2, 1] = V + 1
        with pytest.raises(abi.LrcnError) as ei:
            h.train_epoch(0, badseq, img, blens, np.array([0]), pdrop, seed=1)
        assert ei.value.code == abi.ERR_ARG
        with pytest.raises(abi.LrcnError):
            h.train_epoch(0, seq, img, blens, np.array([6]), pdrop, seed=1)   # order entry outside [0, n_batches)


def test_sticky_error_state_and_adam_update_guard():
    with open_handle(16, 16, 16, 40, 4, 3, abi.PREC_FP32) as h:
        h.load_features(0, np.arange(1, 9), synth.features(8))
        tok = synth.tokens(3, 4, 40)
        h.grad(0, np.arange(1, 5), tok)
        h.adam_update()  # single GPU: fine
        with pytest.raises(abi.LrcnError) as ei:   # argument errors are NOT sticky
            h.loss(0, np.array([1, 2, 3, 999]), tok)
        assert ei.value.code == abi.ERR_MISSING
        s, n = h.loss(0, np.arange(1, 5), tok)
        assert n == 16 and np.isfinite(s)


def test_errors_are_loud():
    E, H1, H2, V, B, l = 16, 16, 16, 40, 4, 3
    with open_handle(E, H1, H2, V, B, l, abi.PREC_FP32) as h:
        tok = synth.tokens(l, B, V)
        with pytest.raises(abi.LrcnError) as ei:
            h.loss(0, np.arange(1, B + 1), tok)
        assert ei.value.code == abi.ERR_STATE  # no features loaded
        h.load_features(0, np.arange(1, 9), synth.features(8))
        with pytest.raises(abi.LrcnError) as ei:
            h.loss(0, np.array([1, 2, 3, 999]), tok)
        assert ei.value.code == abi.ERR_MISSING and "missing features" in str(ei.value)
        bad = tok.copy()
        bad[0, 0] = V + 1
        with pytest.raises(abi.LrcnError):
            h.loss(0, np.arange(1, B + 1), bad)
    with pytest.raises(abi.LrcnError):
        abi.Handle(abi.default_config(embed=8, hidden1=8, hidden2=7, vocab=20, max_batch=2, max_len=2, precision=abi.PREC_FP32))


# ----------------------------------------------------------------------------- generation
@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("K", [1, 3, 5])
def test_beam_search_matches_oracle(prec, K):
    E, H1, H2, V, n_img, nword = 64, 64, 64, 200, 24, 12
    model = synth.initweights([H1, H2], V, E, seed=7)
    model = [w * np.float32(6) if w.shape[0] > 1 else w for w in model]
    model[8][0, O.EOS - 1] = 0.65  # bias eos so that decode lengths vary
    feats = synth.features(n_img, seed=9) * np.float32(100)
    ids = np.arange(1, n_img + 1, dtype=np.int64)
    with open_handle(E, H1, H2, V, 4, 3, prec, gen_rows=40) as h:  # 40 rows -> several chunks at K=3,5
        h.set_model(model)
        h.load_features(1, ids, feats)
        toks, lens, prob, lps = h.beam_search(1, ids, K, nword)
    same = 0
    assert lens.mean() >= 5 and lens.max() > lens.min(), "decodes too short to exercise the recurrent state"
    for i in range(n_img):
        trace = []
        ref_t, ref_p = O.generate(model, feats[i], nword, K, trace=trace)
        got = toks[i, :lens[i]].tolist()
        if got == ref_t:
            same += 1
            assert abs(prob[i] - ref_p) <= 2e-4 * ref_p
            np.testing.assert_allclose(lps[i, :lens[i] - 1], np.array(trace[0], np.float32), rtol=1e-4, atol=1e-4)
        assert got[0] == O.BOS and len(got) <= nword + 2
    assert same >= int(np.ceil(0.99 * n_img)), f"only {same}/{n_img} captions identical"


def test_beam_search_many_rows_path_matches_small_batches_and_oracle():
    # > 512 rows in flight switches generation to the throughput path ([x|h] GEMM operands, elementwise cell kernel)
    if abi.PREC_BF16X3 not in PRECS:
        pytest.skip("tcgen05 path only")
    E, H1, H2, V, n_img, nword, K = 64, 64, 64, 200, 200, 12, 3
    model = synth.initweights([H1, H2], V, E, seed=7)
    model = [w * np.float32(6) if w.shape[0] > 1 else w for w in model]
    model[8][0, O.EOS - 1] = 0.65
    feats = synth.features(n_img, seed=9) * np.float32(100)
    ids = np.arange(1, n_img + 1, dtype=np.int64)
    res = []
    for gen_rows in (900, 60):
        with open_handle(E, H1, H2, V, 4, 3, abi.PREC_BF16X3, gen_rows=gen_rows) as h:
            h.set_model(model)
            h.load_features(1, ids, feats)
            res.append(h.beam_search(1, ids, K, nword))
    (ta, la, pa, _), (tb, lb, pb, _) = res
    same = sum(int(la[i] == lb[i] and (ta[i, :la[i]] == tb[i, :lb[i]]).all()) for i in range(n_img))
    assert same >= int(np.ceil(0.99 * n_img)), f"wide vs narrow path: only {same}/{n_img} captions identical"
    ok = 0
    for i in range(24):
        ref_t, ref_p = O.generate(model, feats[i], nword, K)
        ok += int(ta[i, :la[i]].tolist() == ref_t)
    assert ok >= 23


def test_host_mirror_train_and_generate_text():
    # the reference-facing host API: minibatch format in, caption text out (lrcn.jl:257-297, 585-642)
    import io
    words = [f"w{k}" for k in range(4, 60)]
    vocab = {"~~": 1, "``": 2, "##": 3}
    vocab.update({w: i + 4 for i, w in enumerate(words)})
    rs = np.random.RandomState(0)
    caps = []
    for n in range(200):
        L = 3 + (n // 50)
        caps.append(((int(rs.randint(1, 33)), [words[rs.randint(len(words))] for _ in range(L)]), L))
    seq = host.minibatch(caps, vocab, 10)
    sequence, input_ids, lengths = seq
    assert len(sequence) == sum(lengths) // 10 and all(len(s) == 10 for s in sequence)
    net = host.LRCN([32, 32], len(vocab), 32, 10, precision=abi.PREC_FP32, max_gen_rows=12)
    model = net.initweights(seed=1)
    feats = {i: synth.features(1, seed=100 + i)[0] for i in range(1, 33)}
    net.load_features(feats, 0)
    net.load_features(feats, 1)
    before = net.average_loss(seq)
    assert abs(before - np.log(len(vocab))) < 0.2
    log = io.StringIO()
    hist = net.train((seq, seq), vocab, epochs=3, pdrop=0.0, out=log)     # train! (lrcn.jl:222-239): train1 + average_loss on both splits
    assert len(hist) == 3 and log.getvalue().count("(:epoch,") == 3
    assert abs(hist[-1][0] - hist[-1][1]) < 1e-5 * hist[-1][0]             # both splits hold the same data here
    after = net.average_loss(seq, per_step=True)                           # the per-batch path agrees with the one-call path
    assert abs(after - hist[-1][0]) < 1e-5 * after
    assert after < before - 0.05
    out, in_out = io.StringIO(), io.StringIO()
    hyp = net.generate(5, vocab, 30, 3, out=out, in_out=in_out)
    assert in_out.getvalue() == "5\n"
    line = out.getvalue()
    assert line.endswith(".\n") and hyp[0] == 2
    with pytest.raises(RuntimeError, match="misssing features"):
        net.generate(9999, vocab, 30, 3, out=out, in_out=in_out)
    net.close()


@pytest.mark.parametrize("prec", PRECS)
def test_golden_fixture_through_the_c_abi(prec):
    """The CUDA path against the committed golden vectors (tests/golden/tiny_train.npz); no oracle code runs here."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "tiny_train.npz"))
    E, H1, H2, V, B, l = [int(x) for x in z["cfg"]]
    m = synth.initweights([H1, H2], V, E, seed=1)
    m = [w * np.float32(3) if w.shape[0] > 1 else w for w in m]
    X = synth.features(B, seed=2) * np.float32(50)
    tok = synth.tokens(l, B, V, seed=3)
    ids = np.arange(1, B + 1, dtype=np.int64)
    with open_handle(E, H1, H2, V, B, l, prec) as h:
        h.set_model(m)
        h.load_features(0, ids, X)
        L = h.grad(0, ids, tok)
        assert abs(L - float(z["loss"])) < 1e-4 * abs(float(z["loss"]))
        for k in range(1, 10):
            assert relerr(h.get_grad(k), z[f"g{k}"]) < 1e-4, k
        for _ in range(2):
            h.train_step(0, ids, tok)
        w2 = h.get_model()
        for k in range(9):
            d_ref = z[f"w2_{k + 1}"] - m[k]
            assert np.linalg.norm((w2[k] - m[k]) - d_ref) < 5e-3 * np.linalg.norm(d_ref) + 1e-9, k
        h.set_model(m)
        toks, lens, prob, _ = h.beam_search(0, ids, 3, 8)
        same = 0
        for i in range(B):
            n = int(z["beam_len"][i])
            if int(lens[i]) == n and toks[i][:n].tolist() == z["beam_tokens"][i][:n].tolist():
                same += 1
                assert abs(prob[i] - z["beam_prob"][i]) <= 1e-4 * abs(z["beam_prob"][i])
        assert same >= B - 1  # an untrained net has near-ties; the bit-exact selection logic is tested on identical probabilities


def test_full_size_properties_flickr30k_config():
    """BASELINE.json configs[1] at full size (E=H=512, V=7731, 256 captions, l=12), where the oracle is too slow to run:
    size-independent properties of the hot path instead (SURVEY section 8c / task section 3)."""
    if abi.PREC_BF16X3 not in PRECS:
        pytest.skip("tcgen05 path only")
    E = H = 512
    V, B, l, n_img = 7731, 256, 12, 512
    T = l + 1
    model = synth.initweights([H, H], V, E, seed=1)
    feats = synth.features(n_img, seed=2)
    ids = np.arange(1, n_img + 1, dtype=np.int64)
    img = synth.image_ids(B, n_img)
    tok = synth.tokens(l, B, V, zipf=True)
    with open_handle(E, H, H, V, B, 28, abi.PREC_BF16X3) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        # (1) reproducibility of the forward pass (split-K partial sums land in any order: not bitwise) and a fixed answer
        #     for Wout = 0, bout = 0: loss = ln V (lrcn.jl:562-580)
        s1, n1 = h.loss(0, img, tok)
        s2, n2 = h.loss(0, img, tok)
        assert abs(s1 - s2) <= 1e-6 * abs(s1) and n1 == n2 == B * T
        m0 = [w.copy() for w in model]
        m0[7][:] = 0
        m0[8][:] = 0
        h.set_model(m0)
        s0, _ = h.loss(0, img, tok)
        assert abs(-s0 / (B * T) - np.log(V)) < 1e-5 * np.log(V)
        # (2) softmax - onehot sums to zero over the vocabulary: so does the output-bias gradient
        h.set_model(model)
        L = h.grad(0, img, tok)
        g = [h.get_grad(k) for k in range(1, 10)]
        assert abs(L - (-s1 / (B * T))) < 1e-6 * abs(L)
        assert abs(g[8].astype(np.float64).sum()) < 1e-4 * np.abs(g[8]).astype(np.float64).sum()
        # every embedding row that is not an input token has exactly zero gradient (dense zero + add-at-index adjoint)
        used = np.zeros(V, bool)
        used[tok.ravel() - 1] = True
        used[O.BOS - 1] = True
        assert not g[6][~used].any() and np.abs(g[6][used]).max() > 0
        # (3) gradients are sums over captions: the gradient of the batch is the mean of the gradients of its two halves
        #     (different tile counts / stream-K decompositions / LSTM tile occupancy on the same kernels)
        ga = [None] * 9
        gb = [None] * 9
        La = h.grad(0, img[:B // 2], np.ascontiguousarray(tok[:, :B // 2]))
        ga = [h.get_grad(k) for k in range(1, 10)]
        Lb = h.grad(0, img[B // 2:], np.ascontiguousarray(tok[:, B // 2:]))
        gb = [h.get_grad(k) for k in range(1, 10)]
        assert abs(0.5 * (La + Lb) - L) < 1e-5 * abs(L)
        for k in range(9):
            assert relerr(0.5 * (ga[k] + gb[k]), g[k]) < 1e-4, k
        # (4) first Adam step moves every weight with a non-negligible gradient by lr (Knet Adam, lrcn.jl:394,402)
        h.grad(0, img, tok)
        g = [h.get_grad(k) for k in range(1, 10)]
        h.train_step(0, img, tok)
        w1 = h.get_model()
        for k in (0, 2, 7):  # step 1: m/(1-b1) = g, v/(1-b2) = g^2  =>  dw = -lr * g / (|g| + eps)
            ga_ = np.abs(g[k].astype(np.float64))
            want = 1e-3 * ga_ / (ga_ + 1e-8)
            got = np.abs(w1[k].astype(np.float64) - model[k].astype(np.float64))
            assert (ga_ > 1e-7).any()
            # fp32 weight ulp ~4e-9; the step recomputes the gradient and partial sums land in any order, so entries that are
            # sums cancelling to ~1e-12 carry percent-level noise: check where the gradient is well above that
            bad = (np.abs(got - want) > 1e-2 * want + 1e-8) & (ga_ > 1e-8)  # |g| ~ eps = 1e-8 and below: dw depends on g to first order, and g carries summation-order noise
            assert bad.sum() == 0, (k, int(bad.sum()), float(np.abs(got - want).max()), got[bad][:4], want[bad][:4], ga_[bad][:4])
