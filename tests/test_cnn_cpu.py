"""CPU checks of the fc7 producer's layouts (no GPU): the fp64 VGG-16 oracle's conv, pool and flatten agree with a naive
loop restatement of the ABI formulas on flat column-major buffers, and the host-side extract_features marshals ids and
the normalisation flag."""
import numpy as np

import lrcn_b200  # noqa: F401
from lrcn_b200 import abi, host
import vgg_oracle as V


def naive_conv(x, w, b, pad):
    """out(y,x,o) = b(o) + sum w(dy,dx,c,o) in(y+dy-p, x+dx-p, c) on flat buffers with the header's offsets."""
    H, W, C, n = x.shape
    kh, kw, cin, cout = w.shape
    xf, wf = x.ravel(order="F"), w.ravel(order="F")
    Ho, Wo = H + 2 * pad - kh + 1, W + 2 * pad - kw + 1
    out = np.zeros(Ho * Wo * cout * n)
    for i in range(n):
        for o in range(cout):
            for xx in range(Wo):
                for y in range(Ho):
                    s = float(b[o])
                    for c in range(C):
                        for dx in range(kw):
                            for dy in range(kh):
                                yi, xi = y + dy - pad, xx + dx - pad
                                if 0 <= yi < H and 0 <= xi < W:
                                    s += wf[dy + kh * dx + kh * kw * c + kh * kw * cin * o] * xf[yi + H * xi + H * W * c + H * W * C * i]
                    out[y + Ho * xx + Ho * Wo * o + Ho * Wo * cout * i] = s
    return out.reshape((Ho, Wo, cout, n), order="F")


def naive_pool(x):
    H, W, C, n = x.shape
    xf = x.ravel(order="F")
    out = np.zeros((H // 2) * (W // 2) * C * n)
    for i in range(n):
        for c in range(C):
            for xx in range(W // 2):
                for y in range(H // 2):
                    out[y + (H // 2) * xx + (H // 2) * (W // 2) * c + (H // 2) * (W // 2) * C * i] = max(
                        xf[(2 * y + a) + H * (2 * xx + d) + H * W * c + H * W * C * i] for a in (0, 1) for d in (0, 1))
    return out.reshape((H // 2, W // 2, C, n), order="F")


def test_oracle_conv_matches_naive_formula():
    rs = np.random.RandomState(0)
    x = np.asfortranarray(rs.standard_normal((5, 6, 3, 2)))
    for k, pad in ((3, 1), (1, 0), (2, 0)):
        w = np.asfortranarray(rs.standard_normal((k, k, 3, 4)))
        b = rs.standard_normal(4)
        assert np.allclose(V.conv(x, w, b, pad), naive_conv(x, w, b, pad), rtol=1e-12, atol=1e-12)


def test_oracle_pool_and_flatten_match_naive_formula():
    rs = np.random.RandomState(1)
    x = np.asfortranarray(rs.standard_normal((6, 4, 3, 2)))
    assert np.array_equal(V.pool(x), naive_pool(x))
    # fc6 is a conv whose kernel covers the whole pooled map: out(o) = b(o) + sum w(dy,dx,c,o) in(dy,dx,c)
    m = np.asfortranarray(rs.standard_normal((3, 3, 5, 2)))
    w = np.asfortranarray(rs.standard_normal((3, 3, 5, 7)))
    b = rs.standard_normal(7)
    out = V.conv(m, w, b, 0)
    assert out.shape == (1, 1, 7, 2)
    flat = w.reshape(-1, 7, order="F").T @ m.reshape(-1, 2, order="F") + b[:, None]
    assert np.allclose(out[0, 0], flat, rtol=1e-12, atol=1e-12)
    assert np.allclose(out, naive_conv(m, w, b, 0), rtol=1e-12, atol=1e-12)


def test_oracle_shapes_and_l1():
    assert V.SHAPES == abi.CNN_SHAPES and V.POOL_AFTER == abi.CNN_POOL_AFTER
    f = np.array([[1.0, 3.0, 0.0], [0.0, 0.0, 0.0]])
    assert np.array_equal(V.l1_normalize(f), [[0.25, 0.75, 0.0], [0.0, 0.0, 0.0]])


class _FakeHandle:
    def __init__(self):
        self.calls = []

    def extract_features(self, images, flags):
        self.calls.append((images.shape, flags))
        n = images.shape[3]
        return np.arange(n * 4096, dtype=np.float32).reshape(n, 4096)

    def set_cnn_param(self, layer, which, a):
        self.calls.append((layer, which, np.shape(a)))


def test_host_extract_features_keeps_id_order_and_passes_the_flag():
    net = host.LRCN.__new__(host.LRCN)
    net.h = _FakeHandle()
    imgs = np.zeros((224, 224, 3, 3), dtype=np.float32, order="F")
    d = net.extract_features(imgs, [42, 7, 19])
    assert list(d) == [42, 7, 19]
    assert d[7][0] == 4096 and d[19][-1] == 3 * 4096 - 1
    net.extract_features(imgs, [1, 2, 3], normalize=False)
    assert [c[1] for c in net.h.calls] == [abi.FEAT_L1, 0]
    net.h.calls.clear()
    net.load_cnn([(np.zeros(s, np.float32), np.zeros(s[3], np.float32)) for s in abi.CNN_SHAPES])
    assert [(c[0], c[1]) for c in net.h.calls] == [(l, w) for l in range(1, 16) for w in (0, 1)]
