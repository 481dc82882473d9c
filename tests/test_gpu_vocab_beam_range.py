"""GPU parity over the whole vocabulary and beam-width range the C ABI accepts: 4 <= V <= 51 192 (lrcn_create: one padded
logits row must fit 200 KiB of shared memory) and 1 <= K <= 11 (lrcn_beam_search).  Which kernel runs depends on V, K and
the row count R; this file puts a case on both sides of every bound, against fp64 references (plain numpy or the oracle).

Top-K selection for beam search, beam_row_topk (csrc/kernels_simt.cu).  Rows are padded to ldV = roundup(V, 8), so they are
always 16-byte aligned.

  kernel                              taken when                                         covered here by
  beam_row_topk4_kernel (warp/row),   R >= TOPK4_MIN_ROWS = 2048, V % 4 == 0, V >= 128   R = 2048 at V = 128, 4096, 11264, 51192;
    KM = 1 / 3 / 5 / 11 for                                                              K = 1..6, 10, 11 (full and partly filled
    K = 1 / 2-3 / 4-5 / 6-11                                                             lists); the 1024-image decode's first steps
  beam_row_topk3_kernel (row in       R < 2048, V % 4 == 0, 4096 < V <= 11264            V = 11264 (static + dynamic shared memory just
    registers, grid = min(R, 444))                                                       under 48 KB); R = 2047 (persistent row loop);
                                                                                         decodes at V = 10000, 660 rows in flight
  beam_row_topk2_kernel (row in       everything else: V <= 4096, V % 4 != 0 (7731),     V = 127, 4096, 4100, 7731, 11268, 51192
    shared memory, grid = min(R,      V > 11264 up to the 200 KiB row (51192), and       (200 KiB dynamic shared memory); R = 2047 and
    1184))                            R >= 2048 with V % 4 != 0 or V < 128               2048 (persistent row loop, shared row reused)
  exact fallback in each kernel       more than 256 candidates >= tau                    all-equal rows, 300 copies of the maximum

Softmax cross-entropy in training, softmax_ce_fused (kernels_simt.cu), nv4 = ceil(ldV / 2048):
  <2> nv4 <= 2 (V <= 4096), <4> nv4 <= 4 (V <= 8192), <6> nv4 <= 6 (V <= 12288), <8> nv4 <= 8 (V <= 16384); above that the
  bf16x3 mode runs softmax_ce_kernel plus a separate colsum for the output-bias gradient, as the fp32 mode always does.
  Covered: V = 4096 / 4097 / 8192 / 8193 / 12288 / 12289 / 16384 / 16385 / 51192 at R = 320 rows, so every fused variant runs
  its persistent row loop with the next-row prefetch (grid = min(R, 296), or min(R, 148) for <6> / <8>).

Beam bookkeeping, beam_advance_kernel (kernels_simt.cu): the per-image selection over K*K candidates (beam_pick) keeps two
64-bit "used" masks; the second is reached from K = 9 (K*K > 64).  Covered by decodes at K = 10 and 11.

Generation at coco_2f dimensions (E = H = 1000, C = 500, V = 10636): per-step LSTM gen kernels up to 512 rows, the wide
[x|h] operand path (ld2 = 2C + H2 = 2000) above.

Bars are those of the other GPU tests (BASELINE.json north_star): token ids bit-exact where the logits around the cut are
distinct, log-probs within 1e-4; loss and the nine gradients within 1e-4 relative; >= 99 % identical captions, path
probability within 2e-4 and token log-probs within 1e-4 on identical captions."""
import os

import numpy as np
import pytest

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, synth
from oracle import lrcn_oracle as O

pytestmark = pytest.mark.gpu

PRECS = [int(x) for x in os.environ.get("LRCN_TEST_PRECS", "0,1").split(",")]  # 0 = fp32 CUDA cores, 1 = bf16x3 tcgen05
RTOL = 1e-4
V_MAX = 51192  # (V + 8) * 4 bytes = 200 KiB


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))


def open_handle(E, H, V, B, l, prec, gen_rows=8, hooks=False):
    cfg = abi.default_config(embed=E, hidden1=H, hidden2=H, vocab=V, max_batch=B, max_len=max(l, 1), max_gen_rows=gen_rows,
                             precision=prec)
    return abi.Handle(cfg, hooks=hooks)


# ----------------------------------------------------------------------------- 1. top-K from logits
TOPK_V = [127, 128, 4096, 4100, 7731, 11264, 11268, V_MAX]
TOPK_R = [48, 2047, 2048]
TOPK_K = [1, 2, 3, 4, 5, 6, 10, 11]


@pytest.fixture(scope="module")
def hook_handle():
    # the hook takes V and R per call: one handle serves every case
    with open_handle(64, 64, 128, 4, 2, abi.PREC_FP32, hooks=True) as h:
        yield h


def planted_logits(V, R, seed):
    """Near-uniform rows (sigma 0.02) with special rows planted at fixed positions; returns (logits, {name: row})."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((R, V), dtype=np.float32)
    x *= np.float32(0.02)
    rows = {}
    x[8:16] = rng.standard_normal((8, V), dtype=np.float32) * np.float32(3)       # peaked
    rows["tie3"] = 16
    x[16, [min(123, V - 3), V // 2 + 1, V - 1]] = 5.0                                # exact three-way tie at the top
    rows["equal"] = 17
    x[17] = 0.25                                                                     # all equal: fallback, answer 1..K
    rows["copies"] = 18                                                              # many copies of the maximum, distinct
    x[18] = rng.uniform(-3, 3, V).astype(np.float32)                                 # values elsewhere: fallback with ties
    x[18, np.sort(rng.choice(V, min(300, V - 16), replace=False))] = 4.0
    x[19, 7] = x[19, 8] = -0.5                                                       # tie far below the top
    x[20, 0] = 9.0                                                                   # winner in column 0
    x[21, V - 1] = 9.0                                                               # winner in the last column (scalar tail if V % 4)
    # the K + 1 largest values (K <= 11) in the columns of ONE thread of the CTA kernels (float4 q = t + 256 i) and of ONE lane
    # of topk4 (float4 q = lane + 32 i), as far as the row reaches; values out of column order
    for r, t, stride in ((22, 5, 4 * 256), (23, 3, 4 * 32)):
        cols = [c for c in (4 * t + stride * i + (i % 4) for i in range(12)) if c < 4 * (V // 4)]
        x[r, cols] = 6.0 + 0.25 * rng.permutation(len(cols)).astype(np.float32)
    x[24] = np.linspace(-3, 3, V, dtype=np.float32)                                  # monotone ramp: the online max rises in every chunk
    x[25] = rng.uniform(-60, 60, V).astype(np.float32)                               # wide range: most exp terms underflow
    return x, rows


def topk_reference(logits, M, block=128):
    """fp64 log-softmax and the first M columns of each row in the order (logit desc, index asc), in row blocks."""
    R, V = logits.shape
    idx = np.empty((R, M), np.int64)
    lp = np.empty((R, M), np.float64)
    for r0 in range(0, R, block):
        blk = logits[r0:r0 + block].astype(np.float64)
        mx = blk.max(1, keepdims=True)
        lse = mx[:, 0] + np.log(np.exp(blk - mx).sum(1))
        part = np.argpartition(-blk, M - 1, axis=1)[:, :M]
        cut = np.take_along_axis(blk, part, 1).min(1)                  # the M-th largest value
        for i in range(blk.shape[0]):
            cand = np.flatnonzero(blk[i] >= cut[i])                   # ascending columns, every tie at the cut included
            order = cand[np.argsort(-blk[i, cand], kind="stable")[:M]]
            idx[r0 + i] = order
            lp[r0 + i] = blk[i, order] - lse[i]
    return idx, lp


@pytest.mark.parametrize("R", TOPK_R)
@pytest.mark.parametrize("V", TOPK_V)
def test_topk_from_logits_at_dispatch_bounds(hook_handle, V, R):
    logits, rows = planted_logits(V, R, seed=V + R)
    parent = np.random.default_rng(R).uniform(0.05, 1.0, R).astype(np.float32)
    Kmax = max(TOPK_K)
    ref_idx, ref_lp = topk_reference(logits, Kmax + 1)
    vals = np.take_along_axis(logits, ref_idx, 1).astype(np.float64)
    worst = 0.0
    for K in TOPK_K:
        tok, sc, lp = hook_handle.test_beam_topk_logits(logits, parent, K)
        want = ref_idx[:, :K] + 1
        # The reference sorts fp32 probabilities (stable: equal ones keep the lower index, lrcn.jl:655-661).  Distinct logits closer
        # than ~4e-7 can round to one probability depending on the last bit of the normaliser, and so can logits closer than the
        # fp32 spacing of their log-prob (x - max) - lse, which is 9.5e-7 once |log-prob| >= 8 (near-uniform rows from V ~ 3000
        # up): both round to the same log-prob, hence the same probability.  Such rows are compared as sets, and skipped when the
        # K-th / (K+1)-th pair itself is that close.  Exact logit ties stay strict.
        gaps = vals[:, :K] - vals[:, 1:K + 1]
        close = np.maximum(5e-7, np.spacing(np.abs(ref_lp[:, :K]).astype(np.float32)).astype(np.float64))
        amb = (gaps > 0) & (gaps < close)
        strict = ~amb.any(1)
        for r in np.flatnonzero(amb.any(1) & ~amb[:, -1]):
            assert sorted(tok[r].tolist()) == sorted(want[r].tolist()), f"V={V} R={R} K={K} row {r}"
        bad = np.flatnonzero(strict & (tok != want).any(1))
        assert bad.size == 0, f"V={V} R={R} K={K} rows {bad[:8].tolist()}: got {tok[bad[0]].tolist()} want {want[bad[0]].tolist()}"
        assert strict.sum() >= 0.97 * R, (V, R, K, int(strict.sum()))
        np.testing.assert_allclose(lp[strict], ref_lp[strict, :K], rtol=1e-4, atol=2e-5, err_msg=f"log-probs V={V} R={R} K={K}")
        np.testing.assert_allclose(sc[strict], np.exp(ref_lp[strict, :K]) * parent[strict, None], rtol=5e-5,
                                   err_msg=f"scores V={V} R={R} K={K}")
        worst = max(worst, float(np.abs(lp[strict] - ref_lp[strict, :K]).max()))
        # planted rows, spelled out
        assert tok[rows["equal"]].tolist() == list(range(1, K + 1))
        tie = sorted([min(123, V - 3), V // 2 + 1, V - 1])
        assert tok[rows["tie3"], :min(K, 3)].tolist() == [c + 1 for c in tie][:min(K, 3)]
        assert tok[20, 0] == 1 and tok[21, 0] == V
        copies = np.flatnonzero(logits[rows["copies"]] == 4.0)
        assert tok[rows["copies"]].tolist() == (copies[:K] + 1).tolist()
    print(f"top-K V={V} R={R}: max |log-prob error| {worst:.2e}")


# ----------------------------------------------------------------------------- 2. softmax-CE variants in training
SMX_V = [4096, 4097,      # <2> | <4>
         8192, 8193,      # <4> | <6>
         12288, 12289,    # <6> | <8>
         16384, 16385,    # <8> | softmax_ce_kernel + colsum
         V_MAX]           # largest vocabulary: 200 KiB row in shared memory


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("V", SMX_V)
def test_loss_and_gradients_at_softmax_variant_bounds(prec, V):
    E = H = 64
    B, l, n_img = 32, 9, 40  # R = 320 rows: at least two rows per CTA in every fused variant
    model = synth.initweights([H, H], V, E, seed=11)
    model = [w * np.float32(3) if w.shape[0] > 1 else w for w in model]
    feats = synth.features(n_img, seed=2) * np.float32(50)
    ids = np.arange(1, n_img + 1, dtype=np.int64)
    img = synth.image_ids(B, n_img, seed=5)
    tok = synth.tokens(l, B, V, seed=3)
    tok[0, :4] = [V, V - 1, V - 2, V - 3]    # targets in the last, partly padded float4 group
    tok[4, 4:8] = [V - 3, V - 2, V - 1, V]
    tok[8, :3] = V
    tok[2, 9:12] = 4                         # the smallest non-special id
    X = feats[img - 1]
    g_ref, L_ref = O.lossgradient(model, O.initstate(model, B), X, list(tok), range(0, l))
    lp_ref = O.token_logps(model, O.initstate(model, B), X, list(tok), range(0, l))
    with open_handle(E, H, V, B, l, prec) as h:
        h.set_model(model)
        h.load_features(0, ids, feats)
        s, n = h.loss(0, img, tok)
        assert n == B * (l + 1) and abs(-s / n - L_ref) < RTOL * abs(L_ref)
        np.testing.assert_allclose(h.token_logps(l, B), lp_ref, rtol=RTOL, atol=2e-5)
        L = h.grad(0, img, tok)
        assert abs(L - L_ref) < RTOL * abs(L_ref)
        errs = [relerr(h.get_grad(k), g_ref[k - 1]) for k in range(1, 10)]
        for k, e in enumerate(errs, 1):
            assert e < RTOL, f"V={V} prec={prec}: gradient of param {k}: {e:.2e}"
        # the output-bias gradient (colpart + colsum in the fused variants, colsum of dA otherwise): softmax - onehot sums to
        # zero over the vocabulary, and the target columns in the padded tail match element by element
        gb, gb_ref = h.get_grad(9)[0].astype(np.float64), g_ref[8][0].astype(np.float64)
        assert abs(gb.sum()) < 1e-4 * np.abs(gb).sum()
        cols = [3, V - 4, V - 3, V - 2, V - 1]
        np.testing.assert_allclose(gb[cols], gb_ref[cols], rtol=RTOL, atol=1e-4 * np.abs(gb_ref[cols]).max())
    print(f"softmax-CE V={V} prec={prec}: max gradient relerr {max(errs):.2e}")


def test_create_accepts_the_largest_vocabulary_only():
    with open_handle(64, 64, V_MAX, 4, 2, abi.PREC_FP32):
        pass
    with pytest.raises(abi.LrcnError) as ei:
        open_handle(64, 64, V_MAX + 1, 4, 2, abi.PREC_FP32)
    assert ei.value.code == abi.ERR_ARG and "shared-memory" in str(ei.value)


# ----------------------------------------------------------------------------- 3. lrcn_beam_search against the oracle
_ORACLE = {}  # (case, image, K, nword) -> (tokens, path probability, token log-probs): shared by both precisions


def oracle_caption(case, model, feat, i, K, nword):
    key = (case, i, K, nword)
    if key not in _ORACLE:
        trace = []
        t, p = O.generate(model, feat, nword, K, trace=trace)
        _ORACLE[key] = (t, p, np.array(trace[0], np.float32))
    return _ORACLE[key]


def check_against_oracle(case, model, feats, images, out, K, nword):
    """>= 99 % of `images` decode to the oracle's caption; identical ones carry its path probability and log-probs.
    Returns the largest relative path-probability error seen."""
    toks, lens, prob, lps = out
    same, worst = 0, 0.0
    for i in images:
        ref_t, ref_p, ref_lp = oracle_caption(case, model, feats[i], i, K, nword)
        got = toks[i, :lens[i]].tolist()
        assert got[0] == O.BOS and len(got) <= nword + 2
        if got == ref_t:
            same += 1
            assert abs(prob[i] - ref_p) <= 2e-4 * ref_p, (case, i, prob[i], ref_p)
            np.testing.assert_allclose(lps[i, :lens[i] - 1], ref_lp, rtol=1e-4, atol=1e-4, err_msg=f"{case} image {i}")
            if ref_p > 0:  # long decodes underflow the fp32 product to 0 in both, as in the reference
                worst = max(worst, abs(float(prob[i]) - float(ref_p)) / float(ref_p))
    assert same >= int(np.ceil(0.99 * len(images))), f"{case} K={K}: only {same}/{len(images)} captions identical"
    return worst


def same_captions(a, b, n):
    (ta, la, _, _), (tb, lb, _, _) = a, b
    return sum(int(la[i] == lb[i] and (ta[i, :la[i]] == tb[i, :lb[i]]).all()) for i in range(n))


def decode(E, V, prec, model, feats, K, nword, gen_rows):
    n = feats.shape[0]
    ids = np.arange(1, n + 1, dtype=np.int64)
    with open_handle(E, E, V, 4, 3, prec, gen_rows=gen_rows) as h:
        h.set_model(model)
        h.load_features(1, ids, feats)
        return h.beam_search(1, ids, K, nword)


# a. beam widths 2..11: topk2 at V = 200 (both precisions), topk3 at V = 10000 (bf16x3); 24 images in chunks of 5
BEAM_K = [2, 4, 6, 8, 10, 11]
SMALL = dict(E=64, V=200, w_eos=0.1, g_bias=0.12, v_scale=0.012)
MID = dict(E=128, V=10000, w_eos=0.07, g_bias=0.12, v_scale=0.05)


def timed_model(c):
    return synth.eos_timed_model([c["E"], c["E"]], c["V"], c["E"], w_eos=c["w_eos"], g_bias=c["g_bias"], v_scale=c["v_scale"])


@pytest.mark.parametrize("K", BEAM_K)
@pytest.mark.parametrize("prec,case", [(p, "small") for p in PRECS] + ([(abi.PREC_BF16X3, "mid")] if abi.PREC_BF16X3 in PRECS else []))
def test_beam_widths_match_oracle(prec, case, K):
    c = SMALL if case == "small" else MID
    nword, n_img = 12, 24
    model = timed_model(c)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    out = decode(c["E"], c["V"], prec, model, feats, K, nword, gen_rows=5 * K)   # 5 images per chunk: five chunks
    lens = out[1]
    assert lens.max() > lens.min() and lens.mean() >= 4, f"decode lengths {lens.tolist()} do not exercise the recurrence"
    worst = check_against_oracle(case, model, feats, range(n_img), out, K, nword)
    print(f"beam {case} prec={prec} K={K}: max path-probability relerr {worst:.2e}")


def test_beam_width_11_wide_path_matches_oracle():
    """660 rows in flight: the wide [x|h] generation path and topk3's persistent row loop (grid 444) at K = 11, where the
    selection over K*K = 121 candidates uses the second 'used' mask of beam_advance_kernel."""
    if abi.PREC_BF16X3 not in PRECS:
        pytest.skip("the wide path is the bf16x3 mode's")
    c, K, nword, n_img = MID, 11, 12, 60
    model = timed_model(c)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    out = decode(c["E"], c["V"], abi.PREC_BF16X3, model, feats, K, nword, gen_rows=n_img * K)
    assert n_img * K > 512 and out[1].max() > out[1].min()
    narrow = decode(c["E"], c["V"], abi.PREC_BF16X3, model, feats, K, nword, gen_rows=4 * K)
    assert same_captions(out, narrow, n_img) >= int(np.ceil(0.99 * n_img))
    check_against_oracle("mid", model, feats, range(n_img), out, K, nword)


# b. vocabularies: configs[1] (V = 7731, topk2 since V % 4 != 0) and the largest ones (topk2, up to 200 KiB of shared memory)
def test_beam_flickr30k_vocab_matches_oracle():
    if abi.PREC_BF16X3 not in PRECS:
        pytest.skip("configs[1] runs in the bf16x3 mode")
    E, V, K, nword, n_img = 512, 7731, 3, 30, 100
    model = synth.eos_timed_model([E, E], V, E)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    out = decode(E, V, abi.PREC_BF16X3, model, feats, K, nword, gen_rows=n_img * K)
    assert out[1].max() > out[1].min() and 4 <= out[1].mean() <= 28
    worst = check_against_oracle("flickr30k", model, feats, range(n_img), out, K, nword)
    print(f"beam V=7731: max path-probability relerr {worst:.2e}")


LARGE = {16385: dict(E=64, V=16385, w_eos=0.05, g_bias=0.06, v_scale=0.012),
         V_MAX: dict(E=64, V=V_MAX, w_eos=0.03, g_bias=0.06, v_scale=0.012)}


@pytest.mark.parametrize("prec", PRECS)
@pytest.mark.parametrize("K", [3, 5])
@pytest.mark.parametrize("V", sorted(LARGE))
def test_beam_large_vocab_matches_oracle(prec, K, V):
    c = LARGE[V]
    nword, n_img = 20, 24
    model = timed_model(c)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    out = decode(c["E"], V, prec, model, feats, K, nword, gen_rows=8 * K)
    assert out[1].max() > out[1].min()
    worst = check_against_oracle(f"v{V}", model, feats, range(n_img), out, K, nword)
    print(f"beam V={V} prec={prec} K={K}: max path-probability relerr {worst:.2e}")


# c. 3072 rows at the start: topk4 and the wide path; compaction takes R below 2048 and topk3 over within the same decode
def test_beam_many_rows_switches_kernels_mid_decode():
    if abi.PREC_BF16X3 not in PRECS:
        pytest.skip("the wide path is the bf16x3 mode's")
    E, V, K, nword, n_img = 512, 10000, 3, 30, 1024
    model = synth.eos_timed_model([E, E], V, E)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    many = decode(E, V, abi.PREC_BF16X3, model, feats, K, nword, gen_rows=n_img * K)
    assert n_img * K >= 2048
    lens = many[1]
    # more than a third of the images end before the longest decode: R = 3 * n_act falls below 2048 on the way
    assert (lens < lens.max()).sum() > n_img - 2047 // K, lens.tolist()
    few = decode(E, V, abi.PREC_BF16X3, model, feats, K, nword, gen_rows=60)  # never wide, never topk4
    assert same_captions(many, few, n_img) >= int(np.ceil(0.99 * n_img))
    worst = check_against_oracle("c3", model, feats, range(0, n_img, 8), many, K, nword)
    print(f"beam 1024 images: max path-probability relerr {worst:.2e}")


# d. coco_2f decode (configs[3]): E = H = 1000, C = 500, V = 10636
@pytest.mark.parametrize("prec", PRECS)
def test_beam_coco_2f_matches_oracle(prec):
    E, V, K, nword, n_img = 1000, 10636, 3, 30, 200
    model = synth.eos_timed_model([E, E], V, E)
    feats = synth.features(n_img, seed=9) * np.float32(100)
    narrow = decode(E, V, prec, model, feats[:100], K, nword, gen_rows=300)   # per-step gen kernels at H = 1000
    wide = decode(E, V, prec, model, feats, K, nword, gen_rows=600)           # 600 rows: the wide path in the bf16x3 mode
    assert narrow[1].max() > narrow[1].min()
    assert same_captions(narrow, wide, 100) >= 99
    worst = check_against_oracle("coco_2f", model, feats, range(100), narrow, K, nword)
    worst = max(worst, check_against_oracle("coco_2f", model, feats, range(100, 200), wide, K, nword))
    print(f"beam coco_2f prec={prec}: max path-probability relerr {worst:.2e}")
