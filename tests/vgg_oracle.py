"""fp64 restatement of VGG-16 up to relu7 (the fc7 producer, include/lrcn_b200.h lrcn_extract_features), used only by
tests.  Inputs and outputs use the ABI's column-major layouts as numpy arrays indexed like Julia:
  images / activations: (H, W, C, n) with element (y, x, c, i);  filters: (kh, kw, Cin, Cout) with (dy, dx, c, o).
torch CPU conv2d / max_pool2d do the arithmetic; the permutations to and from torch's NCHW / OIHW are spelled out here."""
import numpy as np
import torch
import torch.nn.functional as F

SHAPES = [(3, 3, 3, 64), (3, 3, 64, 64), (3, 3, 64, 128), (3, 3, 128, 128), (3, 3, 128, 256), (3, 3, 256, 256),
          (3, 3, 256, 256), (3, 3, 256, 512), (3, 3, 512, 512), (3, 3, 512, 512), (3, 3, 512, 512), (3, 3, 512, 512),
          (3, 3, 512, 512), (7, 7, 512, 4096), (1, 1, 4096, 4096)]
POOL_AFTER = (2, 4, 7, 10, 13)  # 1-based layers followed by a 2x2 stride-2 max-pool


def _to_torch(x):   # (H, W, C, n) -> (n, C, H, W)
    return torch.from_numpy(np.asarray(x, np.float64)).permute(3, 2, 0, 1)


def _from_torch(t):  # (n, C, H, W) -> (H, W, C, n)
    return t.permute(2, 3, 1, 0).contiguous().numpy()


def conv(x, w, b, pad):
    """out(y,x,o) = b(o) + sum_{dy,dx,c} w(dy,dx,c,o) in(y+dy-pad, x+dx-pad, c): cross-correlation with zero padding."""
    wt = torch.from_numpy(np.asarray(w, np.float64)).permute(3, 2, 0, 1)  # (kh, kw, Cin, Cout) -> (Cout, Cin, kh, kw)
    bt = torch.from_numpy(np.asarray(b, np.float64).reshape(-1))
    return _from_torch(F.conv2d(_to_torch(x), wt, bt, padding=pad))


def pool(x):
    return _from_torch(F.max_pool2d(_to_torch(x), 2, 2))


def relu(x):
    return np.maximum(x, 0.0)


def vgg16(images, params):
    """images (224, 224, 3, n); params: 15 (filter, bias) pairs.  Returns (the 15 pre-ReLU layer outputs as (H, W, Cout, n),
    relu7 as an n x 4096 array)."""
    acts = []
    x = np.asarray(images, np.float64)
    for layer, (w, b) in enumerate(params, start=1):
        a = conv(x, w, b, 1 if layer <= 13 else 0)
        acts.append(a)
        x = relu(a)
        if layer in POOL_AFTER:
            x = pool(x)
    return acts, np.ascontiguousarray(x[0, 0].T)


def l1_normalize(feats):
    """f /= sum(f) per row; a zero row stays zero."""
    s = feats.sum(axis=1, keepdims=True)
    return np.where(s > 0, feats / np.where(s > 0, s, 1.0), 0.0)


def he_params(seed=0, bias_scale=0.05):
    """He-initialised filters (std sqrt(2 / fan_in)) and small random biases, float32."""
    rs = np.random.RandomState(seed)
    out = []
    for kh, kw, cin, cout in SHAPES:
        w = (rs.standard_normal((kh, kw, cin, cout)) * np.sqrt(2.0 / (kh * kw * cin))).astype(np.float32)
        out.append((np.asfortranarray(w), (rs.standard_normal(cout) * bias_scale).astype(np.float32)))
    return out


def random_images(n, seed=1):
    return np.asfortranarray(np.random.RandomState(seed).standard_normal((224, 224, 3, n)).astype(np.float32))
