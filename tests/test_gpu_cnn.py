"""GPU tests of the fc7 producer (VGG-16 up to relu7, lrcn_extract_features) against the fp64 oracle (tests/vgg_oracle.py),
both precisions (LRCN_TEST_PRECS).  Bars: weights round-trip bit-exactly; every layer's pre-ReLU output and relu7 within
1e-4 relative (Frobenius); chunked extraction equals per-slice calls (1e-6 in fp32, see same_tol); >= 99 % identical
captions downstream."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, synth
import vgg_oracle as V

pytestmark = pytest.mark.gpu

PRECS = [int(x) for x in os.environ.get("LRCN_TEST_PRECS", "0,1").split(",")]
RTOL = 1e-4
NGPU = torch.cuda.device_count() if torch.cuda.is_available() else 0


def relerr(a, b):
    return float(np.linalg.norm(np.asarray(a, np.float64) - np.asarray(b, np.float64)) / (np.linalg.norm(np.asarray(b, np.float64)) + 1e-30))


def open_handle(prec, **kw):
    cfg = abi.default_config(embed=64, hidden1=64, hidden2=64, vocab=300, max_batch=4, max_len=8, max_gen_rows=12, precision=prec, **kw)
    return abi.Handle(cfg, hooks=True)


def load_cnn(h, params):
    for layer, (w, b) in enumerate(params, start=1):
        h.set_cnn_param(layer, 0, w)
        h.set_cnn_param(layer, 1, b)


@pytest.fixture(scope="module")
def params():
    return V.he_params(seed=0)


@pytest.fixture(scope="module")
def reference(params):
    images = V.random_images(3, seed=1)
    acts, relu7 = V.vgg16(images, params)
    return images, acts, relu7


@pytest.fixture(scope="module", params=PRECS)
def net(request, params):
    with open_handle(request.param) as h:
        load_cnn(h, params)
        yield request.param, h


def test_weights_round_trip_bit_exact(net, params):
    _, h = net
    for layer, (w, b) in enumerate(params, start=1):
        assert np.array_equal(h.get_cnn_param(layer, 0), w), layer
        assert np.array_equal(h.get_cnn_param(layer, 1), b), layer


def test_error_codes(net):
    prec, h = net
    lib, hh = h.lib, h._h
    w = np.zeros(3 * 3 * 3 * 64, np.float32)
    ptr = w.ctypes.data_as(C.POINTER(C.c_float))

    def dims(*d):
        return np.array(d, dtype=np.int64).ctypes.data_as(C.POINTER(C.c_int64))

    assert lib.lrcn_set_cnn_param(hh, 1, 0, ptr, dims(3, 3, 64, 3)) == abi.ERR_ARG       # wrong dims
    assert lib.lrcn_set_cnn_param(hh, 1, 1, ptr, dims(64, 1, 1, 2)) == abi.ERR_ARG
    assert lib.lrcn_set_cnn_param(hh, 0, 0, ptr, dims(3, 3, 3, 64)) == abi.ERR_ARG       # layer out of range
    assert lib.lrcn_set_cnn_param(hh, 16, 0, ptr, dims(3, 3, 3, 64)) == abi.ERR_ARG
    assert lib.lrcn_set_cnn_param(hh, 1, 2, ptr, dims(3, 3, 3, 64)) == abi.ERR_ARG       # which out of range
    assert lib.lrcn_set_cnn_param(hh, 1, 0, None, dims(3, 3, 3, 64)) == abi.ERR_ARG      # null data / dims
    assert lib.lrcn_set_cnn_param(hh, 1, 0, ptr, None) == abi.ERR_ARG
    assert lib.lrcn_get_cnn_param(hh, 14, 0, ptr, dims(7, 7, 512, 4095)) == abi.ERR_ARG
    img = np.zeros((224, 224, 3, 1), np.float32, order="F")
    out = np.zeros((1, 4096), np.float32)
    ip, op = img.ctypes.data_as(C.POINTER(C.c_float)), out.ctypes.data_as(C.POINTER(C.c_float))
    assert lib.lrcn_extract_features(hh, ip, 0, 0, op) == abi.ERR_ARG                    # n <= 0
    assert lib.lrcn_extract_features(hh, ip, -2, 0, op) == abi.ERR_ARG
    assert lib.lrcn_extract_features(hh, None, 1, 0, op) == abi.ERR_ARG
    assert lib.lrcn_extract_features(hh, ip, 1, 0, None) == abi.ERR_ARG
    assert lib.lrcn_extract_features(hh, ip, 1, 6, op) == abi.ERR_ARG                    # unknown flag
    # a fresh handle: get before set and extraction before all 30 tensors are set are state errors
    with open_handle(prec) as g:
        assert g.lib.lrcn_get_cnn_param(g._h, 1, 0, ptr, dims(3, 3, 3, 64)) == abi.ERR_STATE
        assert g.lib.lrcn_extract_features(g._h, ip, 1, 0, op) == abi.ERR_STATE
        for layer, s in enumerate(abi.CNN_SHAPES, start=1):
            g.set_cnn_param(layer, 0, np.zeros(s, np.float32))
            if layer != 9:
                g.set_cnn_param(layer, 1, np.zeros(s[3], np.float32))
        assert g.lib.lrcn_extract_features(g._h, ip, 1, 0, op) == abi.ERR_STATE
        assert g.lib.lrcn_test_cnn_activation(g._h, 1, op, 1) == abi.ERR_STATE            # nothing extracted yet
        g.set_cnn_param(9, 1, np.zeros(512, np.float32))
        g.extract_features(img)
        act = np.zeros(224 * 224 * 64 * 2, np.float32)
        assert g.lib.lrcn_test_cnn_activation(g._h, 1, act.ctypes.data_as(C.POINTER(C.c_float)), 2) == abi.ERR_ARG  # n differs
        assert g.lib.lrcn_test_cnn_activation(g._h, 0, op, 1) == abi.ERR_ARG
        g.extract_features(np.zeros((224, 224, 3, 17), np.float32, order="F"))             # two chunks
        assert g.lib.lrcn_test_cnn_activation(g._h, 15, op, 17) == abi.ERR_STATE


def test_conv1_1_delta_filter_pins_orientation_padding_and_channels(net, params):
    prec, h = net
    w = np.zeros((3, 3, 3, 64), np.float32, order="F")
    w[0, 2, 1, 5] = 1.0  # out(y, x, 5) = in(y - 1, x + 1, 1)
    h.set_cnn_param(1, 0, w)
    h.set_cnn_param(1, 1, np.zeros(64, np.float32))
    try:
        imgs = V.random_images(2, seed=7)
        h.extract_features(imgs)
        a = h.test_cnn_activation(1, 2)
    finally:
        h.set_cnn_param(1, 0, params[0][0])
        h.set_cnn_param(1, 1, params[0][1])
    want = np.zeros((224, 224, 2), np.float32)
    want[1:, :-1, :] = imgs[:-1, 1:, 1, :]
    # fp32: the input itself; bf16x3: its hi + lo split (16 significant bits); the padding and the other channels exactly 0
    assert np.array_equal(a[:, :, 5, :] == 0, want == 0)
    np.testing.assert_allclose(a[:, :, 5, :], want, rtol=0 if prec == abi.PREC_FP32 else 2.0 ** -16, atol=0)
    a[:, :, 5, :] = 0
    assert not a.any()


def test_every_layer_and_relu7_match_the_fp64_oracle(net, reference):
    prec, h = net
    images, acts, relu7 = reference
    feats = h.extract_features(images)
    errs = []
    for layer in range(1, 16):
        errs.append(relerr(h.test_cnn_activation(layer, 3), acts[layer - 1]))
    errs.append(relerr(feats, relu7))
    print(f"precision {prec}: per-layer relerr " + " ".join(f"{e:.2e}" for e in errs))
    assert max(errs) < RTOL, errs


def same_tol(prec):
    """Two extractions of the same images, e.g. with different chunk boundaries, run GEMMs with schedules chosen from the
    chunk's pixel count (tile shape, split-K) and split-K partial sums added in arrival order: fp32 results differ in the
    last bits.  In bf16x3 mode every layer's input is split again into bf16 hi + lo, which turns a last-bit difference into
    one of the split's own size (2^-17 relative), so there the bar is the parity bar."""
    return 1e-6 if prec == abi.PREC_FP32 else RTOL


def test_chunked_extraction_equals_per_slice_calls(net):
    prec, h = net
    imgs = V.random_images(40, seed=3)
    whole = h.extract_features(imgs)
    parts = np.concatenate([h.extract_features(imgs[..., a:b]) for a, b in ((0, 7), (7, 23), (23, 40))])
    err = relerr(whole, parts)
    print(f"precision {prec}: chunked vs per-slice relerr {err:.2e}")
    assert err < same_tol(prec)


def test_l1_normalisation_and_all_zero_rows(net, params):
    _, h = net
    imgs = V.random_images(5, seed=4)
    raw = h.extract_features(imgs)
    assert np.array_equal(raw, np.maximum(h.test_cnn_activation(15, 5)[0, 0].T, 0))  # relu7 of this call's fc7
    l1 = h.extract_features(imgs, abi.FEAT_L1)
    raw = np.maximum(h.test_cnn_activation(15, 5)[0, 0].T, 0).astype(np.float64)
    assert (raw.sum(1) > 0).all()
    assert relerr(l1, raw / raw.sum(1, keepdims=True)) < 1e-6
    h.set_cnn_param(15, 1, np.full(4096, -1e6, np.float32))
    try:
        z = h.extract_features(imgs, abi.FEAT_L1)
    finally:
        h.set_cnn_param(15, 1, params[14][1])
    assert np.isfinite(z).all() and not z.any()


def test_extracted_features_caption_like_oracle_features(net, reference):
    prec, h = net
    images, _, relu7 = reference
    feats = h.extract_features(images)
    E, H1, H2, Vs = 64, 64, 64, 300
    model = [w * np.float32(3) if w.shape[0] > 1 else w for w in synth.initweights([H1, H2], Vs, E, seed=1)]
    ids = np.arange(1, len(feats) + 1, dtype=np.int64)
    h.set_model(model)
    h.load_features(0, ids, feats)
    h.load_features(1, ids, relu7.astype(np.float32))
    ours = h.beam_search(0, ids, 3, 8)
    ref = h.beam_search(1, ids, 3, 8)
    same = sum(ours[0][i, :ours[1][i]].tolist() == ref[0][i, :ref[1][i]].tolist() for i in range(len(ids)))
    assert same >= 0.99 * len(ids), (same, len(ids))


@pytest.mark.skipif(NGPU < 2, reason="needs >= 2 GPUs on one node")
@pytest.mark.parametrize("prec", PRECS)
def test_group_handle_matches_one_gpu(prec, params):
    imgs = V.random_images(21, seed=5)
    with open_handle(prec) as h:
        load_cnn(h, params)
        one = h.extract_features(imgs, abi.FEAT_L1)
    cfg = abi.default_config(embed=64, hidden1=64, hidden2=64, vocab=300, max_batch=4, max_len=8, max_gen_rows=12, precision=prec, n_gpus=2)
    cfg.device_ids[0], cfg.device_ids[1] = 0, 1
    with abi.Handle(cfg) as g:
        load_cnn(g, params)
        assert np.array_equal(g.get_cnn_param(14, 0), params[13][0])
        grp = g.extract_features(imgs, abi.FEAT_L1)
    assert relerr(grp, one) < same_tol(prec)
