"""ctypes binding of liblrcn_b200.so -- the executable mirror of the Julia `ccall` shim
(julia/lrcn_b200.jl).  Every symbol declared in include/lrcn_b200.h is bound here with the same
argument order.  There is no fallback: if the library is missing, loading raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblrcn_b200.so")            # the product: include/lrcn_b200.h
TEST_LIB_PATH = os.path.join(_HERE, "liblrcn_b200_test.so")  # + kernel-level test hooks: include/lrcn_b200_testhooks.h
ABI_VERSION = 2

PREC_FP32, PREC_BF16X3 = 0, 1
OK, ERR_ARG, ERR_CUDA, ERR_NCCL, ERR_MISSING, ERR_STATE = 0, 1, 2, 3, 4, 5
COMM_ID_BYTES = 128
P2P_BLOB_BYTES = 512

# VGG-16 up to fc7 (include/lrcn_b200.h, lrcn_set_cnn_param): filter shapes kh x kw x Cin x Cout of layers 1..15 and the
# spatial size of each layer's output
CNN_LAYERS, CNN_IMAGE, FEAT_L1 = 15, 224, 1
CNN_SHAPES = [(3, 3, 3, 64), (3, 3, 64, 64), (3, 3, 64, 128), (3, 3, 128, 128), (3, 3, 128, 256), (3, 3, 256, 256),
              (3, 3, 256, 256), (3, 3, 256, 512), (3, 3, 512, 512), (3, 3, 512, 512), (3, 3, 512, 512), (3, 3, 512, 512),
              (3, 3, 512, 512), (7, 7, 512, 4096), (1, 1, 4096, 4096)]
CNN_HOUT = [224, 224, 112, 112, 56, 56, 56, 28, 28, 28, 14, 14, 14, 1, 1]
CNN_POOL_AFTER = (2, 4, 7, 10, 13)  # 2x2 max-pool after conv1_2, conv2_2, conv3_3, conv4_3, conv5_3


def cnn_dims(layer, which):
    if not 1 <= layer <= CNN_LAYERS or which not in (0, 1):
        raise ValueError(f"CNN layer {layer} / which {which} out of range")
    s = CNN_SHAPES[layer - 1]
    return s if which == 0 else (s[3], 1, 1, 1)


class LrcnError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liblrcn_b200 error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("embed", "hidden1", "hidden2", "vocab", "max_batch", "max_len",
                                         "max_gen_rows", "device", "precision", "use_graphs")] + \
               [(n, C.c_double) for n in ("lr", "beta1", "beta2", "eps")] + \
               [("n_gpus", C.c_int32), ("device_ids", C.c_int32 * 8)]


_p = C.POINTER
_f32p, _i64p, _i32p, _f64p = _p(C.c_float), _p(C.c_int64), _p(C.c_int32), _p(C.c_double)
_H = C.c_void_p

# name -> (restype, argtypes); mirrors include/lrcn_b200.h one to one
SIGNATURES = {
    "lrcn_abi_version": (C.c_int, []),
    "lrcn_last_error": (C.c_char_p, []),
    "lrcn_config_default": (C.c_int, [_p(Config)]),
    "lrcn_create": (C.c_int, [_p(Config), _p(_H)]),
    "lrcn_destroy": (C.c_int, [_H]),
    "lrcn_param_shape": (C.c_int, [_H, C.c_int, _i64p, _i64p]),
    "lrcn_set_param": (C.c_int, [_H, C.c_int, _f32p, C.c_int64, C.c_int64]),
    "lrcn_get_param": (C.c_int, [_H, C.c_int, _f32p, C.c_int64, C.c_int64]),
    "lrcn_get_grad": (C.c_int, [_H, C.c_int, _f32p, C.c_int64, C.c_int64]),
    "lrcn_get_adam_state": (C.c_int, [_H, C.c_int, C.c_int, _f32p, C.c_int64, C.c_int64]),
    "lrcn_set_adam_state": (C.c_int, [_H, C.c_int, C.c_int, _f32p, C.c_int64, C.c_int64]),
    "lrcn_get_adam_step": (C.c_int, [_H, _i64p]),
    "lrcn_set_adam_step": (C.c_int, [_H, C.c_int64]),
    "lrcn_load_features": (C.c_int, [_H, C.c_int, _i64p, _f32p, C.c_int64]),
    "lrcn_loss": (C.c_int, [_H, C.c_int, _i64p, _i64p, C.c_int, C.c_int, _f64p, _i64p]),
    "lrcn_grad": (C.c_int, [_H, C.c_int, _i64p, _i64p, C.c_int, C.c_int, C.c_float, C.c_uint64, _f64p]),
    "lrcn_adam_update": (C.c_int, [_H]),
    "lrcn_train_step": (C.c_int, [_H, C.c_int, _i64p, _i64p, C.c_int, C.c_int, C.c_float, C.c_uint64, _f64p]),
    "lrcn_train_epoch": (C.c_int, [_H, C.c_int, _i64p, C.c_int64, _i64p, _i64p, C.c_int64, C.c_int, _i64p, C.c_int64, C.c_float, C.c_uint64,
                                   _f64p, _i64p]),
    "lrcn_loss_epoch": (C.c_int, [_H, C.c_int, _i64p, C.c_int64, _i64p, _i64p, C.c_int64, C.c_int, _f64p, _i64p]),
    "lrcn_get_token_logps": (C.c_int, [_H, _f32p, C.c_int64]),
    "lrcn_stage_batch": (C.c_int, [_H, C.c_int, C.c_int, _i64p, _i64p, C.c_int, C.c_int]),
    "lrcn_train_step_staged": (C.c_int, [_H, C.c_int, C.c_float, C.c_uint64, _f64p]),
    "lrcn_beam_search": (C.c_int, [_H, C.c_int, _i64p, C.c_int64, C.c_int, C.c_int, _i64p, _i32p, _f32p, _f32p]),
    "lrcn_set_cnn_param": (C.c_int, [_H, C.c_int, C.c_int, _f32p, _i64p]),
    "lrcn_get_cnn_param": (C.c_int, [_H, C.c_int, C.c_int, _f32p, _i64p]),
    "lrcn_extract_features": (C.c_int, [_H, _f32p, C.c_int64, C.c_int, _f32p]),
    "lrcn_checkpoint_save": (C.c_int, [_H, C.c_char_p, C.c_int, C.c_char_p, C.c_int64]),
    "lrcn_checkpoint_load": (C.c_int, [_H, C.c_char_p, _i32p, C.c_char_p, C.c_int64, _i64p]),
    "lrcn_comm_unique_id": (C.c_int, [C.c_char_p]),
    "lrcn_comm_init": (C.c_int, [_H, C.c_char_p, C.c_int, C.c_int]),
    "lrcn_p2p_export": (C.c_int, [_H, C.c_char_p]),
    "lrcn_p2p_import": (C.c_int, [_H, C.c_char_p, C.c_int, C.c_int]),
    "lrcn_sync": (C.c_int, [_H]),
    "lrcn_timer_start": (C.c_int, [_H]),
    "lrcn_timer_stop": (C.c_int, [_H, _f32p]),
    "lrcn_kernel_launches": (C.c_int, [_H, _i64p]),
    "lrcn_flush_l2": (C.c_int, [_H]),
    "lrcn_get_trace": (C.c_int, [_H, _p(C.c_uint64), C.c_int64]),
    "lrcn_time_kernel": (C.c_int, [_H, C.c_char_p, C.c_int, _f32p, _f64p, _f64p]),
}

# kernel-level test hooks: exported by liblrcn_b200_test.so only
TEST_SIGNATURES = {
    "lrcn_test_mma_rate": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "lrcn_test_gemm_time": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p]),
    "lrcn_test_gemm": (C.c_int, [_H, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p, C.c_int, _f32p]),
    "lrcn_test_beam_select": (C.c_int, [_H, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, _i64p, _i32p, _f32p]),
    "lrcn_test_beam_topk_logits": (C.c_int, [_H, _f32p, _f32p, C.c_int, C.c_int, C.c_int, _i64p, _f32p, _f32p]),
    "lrcn_test_cnn_activation": (C.c_int, [_H, C.c_int, _f32p, C.c_int64]),
}

_lib = None
_test_lib = None


def load():
    """Load liblrcn_b200.so (built in-tree by __graft_entry__.build()).  Raises if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FileNotFoundError(f"{LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`. "
                                    "The LRCN hot path has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def load_test():
    """Load liblrcn_b200_test.so: the product objects plus the kernel-level test hooks (tests only)."""
    global _test_lib
    if _test_lib is None:
        if not os.path.exists(TEST_LIB_PATH):
            raise FileNotFoundError(f"{TEST_LIB_PATH} is not built; run `python -c 'import __graft_entry__ as g; g.build()'`.")
        lib = C.CDLL(TEST_LIB_PATH)
        for name, (res, args) in {**SIGNATURES, **TEST_SIGNATURES}.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _test_lib = lib
    return _test_lib


_last_lib = None  # the library called last (each of the two has its own thread-local error message)


class _Lib:
    """Thin proxy over a CDLL that remembers which library was called last, so check() reads the right message."""

    def __init__(self, lib):
        object.__setattr__(self, "_lib", lib)

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        lib = self._lib

        def call(*a):
            global _last_lib
            _last_lib = lib
            return fn(*a)

        object.__setattr__(self, name, call)
        return call


def check(rc):
    if rc != OK:
        lib = _last_lib or load()
        raise LrcnError(rc, lib.lrcn_last_error().decode("utf-8", "replace"))


def _f32(a):
    return a.ctypes.data_as(_f32p)


def _i64(a):
    return a.ctypes.data_as(_i64p)


def default_config(**kw) -> Config:
    cfg = Config()
    check(_Lib(load()).lrcn_config_default(C.byref(cfg)))
    for k, v in kw.items():
        if not hasattr(cfg, k):
            raise AttributeError(k)
        setattr(cfg, k, v)
    return cfg


class Handle:
    """Owns one lrcn_handle: one GPU, or (cfg.n_gpus > 1) a single-process data-parallel group.
    hooks=True binds the handle to liblrcn_b200_test.so so that the test_* methods are available."""

    def __init__(self, cfg: Config, hooks: bool = False):
        self.lib = _Lib(load_test() if hooks else load())
        self.cfg = cfg
        self._h = _H()
        check(self.lib.lrcn_create(C.byref(cfg), C.byref(self._h)))

    def close(self):
        if self._h:
            self.lib.lrcn_destroy(self._h)
            self._h = _H()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # ---- weights
    def param_shape(self, idx):
        r, c = C.c_int64(), C.c_int64()
        check(self.lib.lrcn_param_shape(self._h, idx, C.byref(r), C.byref(c)))
        return int(r.value), int(c.value)

    def set_param(self, idx, w):
        w = np.asfortranarray(w, dtype=np.float32)
        check(self.lib.lrcn_set_param(self._h, idx, _f32(w), w.shape[0], w.shape[1]))

    def _get(self, fn, idx, *pre):
        r, c = self.param_shape(idx)
        out = np.empty((r, c), dtype=np.float32, order="F")
        check(fn(self._h, idx, *pre, _f32(out), r, c))
        return out

    def get_param(self, idx):
        return self._get(self.lib.lrcn_get_param, idx)

    def get_grad(self, idx):
        return self._get(self.lib.lrcn_get_grad, idx)

    def get_adam_state(self, idx, which):
        return self._get(self.lib.lrcn_get_adam_state, idx, which)

    def set_adam_state(self, idx, which, a):
        a = np.asfortranarray(a, dtype=np.float32)
        check(self.lib.lrcn_set_adam_state(self._h, idx, which, _f32(a), a.shape[0], a.shape[1]))

    def get_adam_step(self):
        t = C.c_int64()
        check(self.lib.lrcn_get_adam_step(self._h, C.byref(t)))
        return int(t.value)

    def set_adam_step(self, t):
        check(self.lib.lrcn_set_adam_step(self._h, int(t)))

    def set_model(self, model):
        for k, w in enumerate(model):
            self.set_param(k + 1, w)

    def get_model(self):
        return [self.get_param(k) for k in range(1, 10)]

    # ---- features
    def load_features(self, split, ids, feats):
        ids = np.ascontiguousarray(ids, dtype=np.int64)
        feats = np.ascontiguousarray(feats, dtype=np.float32)
        assert feats.shape == (len(ids), 4096)
        check(self.lib.lrcn_load_features(self._h, split, _i64(ids), _f32(feats), len(ids)))

    # ---- steps
    @staticmethod
    def _batch(image_ids, tokens):
        image_ids = np.ascontiguousarray(image_ids, dtype=np.int64)
        tokens = np.ascontiguousarray(tokens, dtype=np.int64)
        if tokens.ndim == 1:
            tokens = tokens.reshape(0, len(image_ids)) if tokens.size == 0 else tokens.reshape(-1, len(image_ids))
        l, B = tokens.shape
        assert B == len(image_ids)
        return image_ids, tokens, l, B

    def loss(self, split, image_ids, tokens):
        ids, tok, l, B = self._batch(image_ids, tokens)
        s, n = C.c_double(), C.c_int64()
        check(self.lib.lrcn_loss(self._h, split, _i64(ids), _i64(tok), l, B, C.byref(s), C.byref(n)))
        return float(s.value), int(n.value)

    def grad(self, split, image_ids, tokens, pdrop=0.0, seed=0):
        ids, tok, l, B = self._batch(image_ids, tokens)
        out = C.c_double()
        check(self.lib.lrcn_grad(self._h, split, _i64(ids), _i64(tok), l, B, pdrop, seed, C.byref(out)))
        return float(out.value)

    def train_step(self, split, image_ids, tokens, pdrop=0.0, seed=0):
        ids, tok, l, B = self._batch(image_ids, tokens)
        out = C.c_double()
        check(self.lib.lrcn_train_step(self._h, split, _i64(ids), _i64(tok), l, B, pdrop, seed, C.byref(out)))
        return float(out.value)

    def train_epoch(self, split, sequence, input_ids, lengths, order=None, pdrop=0.0, seed=0):
        """One epoch of train steps with the batches staged on the device (lrcn_train_epoch).  sequence: [n_rows][B] time-major
        tokens (1-based), input_ids: [n_batches][B], lengths: [n_batches] rows per batch, order: batch indices to run.
        Returns the per-step losses in execution order (batches longer than max_len are skipped)."""
        seq = np.ascontiguousarray(sequence, dtype=np.int64)
        ids = np.ascontiguousarray(input_ids, dtype=np.int64)
        lens = np.ascontiguousarray(lengths, dtype=np.int64)
        if ids.ndim != 2 or (seq.size and (seq.ndim != 2 or seq.shape[1] != ids.shape[1])) or lens.shape != (ids.shape[0],):
            raise ValueError("sequence [n_rows][B], input_ids [n_batches][B], lengths [n_batches] expected")
        n_batches, B = ids.shape
        n_rows = seq.shape[0] if seq.size else 0
        if n_rows == 0:
            seq = np.zeros((1, B), dtype=np.int64)
        ordr = None if order is None else np.ascontiguousarray(order, dtype=np.int64)
        n_order = 0 if ordr is None else len(ordr)
        losses = np.zeros(max(n_order if ordr is not None else n_batches, 1), dtype=np.float64)
        steps = C.c_int64()
        check(self.lib.lrcn_train_epoch(self._h, split, _i64(seq), n_rows, _i64(ids), _i64(lens), n_batches, B,
                                        _i64(ordr) if n_order else None, n_order, pdrop, seed,
                                        losses.ctypes.data_as(_f64p), C.byref(steps)))
        return losses[:steps.value].tolist()

    def loss_epoch(self, split, sequence, input_ids, lengths):
        """Sum of target log-probs and token count over all batches of a split in one call (lrcn_loss_epoch)."""
        seq = np.ascontiguousarray(sequence, dtype=np.int64)
        ids = np.ascontiguousarray(input_ids, dtype=np.int64)
        lens = np.ascontiguousarray(lengths, dtype=np.int64)
        n_batches, B = ids.shape
        n_rows = seq.shape[0] if seq.size else 0
        if n_rows == 0:
            seq = np.zeros((1, B), dtype=np.int64)
        s, n = C.c_double(), C.c_int64()
        check(self.lib.lrcn_loss_epoch(self._h, split, _i64(seq), n_rows, _i64(ids), _i64(lens), n_batches, B, C.byref(s), C.byref(n)))
        return float(s.value), int(n.value)

    def adam_update(self):
        check(self.lib.lrcn_adam_update(self._h))

    def token_logps(self, l, B):
        out = np.empty((l + 1, B), dtype=np.float32)
        check(self.lib.lrcn_get_token_logps(self._h, _f32(out), out.size))
        return out

    def stage_batch(self, slot, split, image_ids, tokens):
        ids, tok, l, B = self._batch(image_ids, tokens)
        check(self.lib.lrcn_stage_batch(self._h, slot, split, _i64(ids), _i64(tok), l, B))

    def train_step_staged(self, slot, pdrop=0.0, seed=0, want_loss=False):
        if want_loss:
            out = C.c_double()
            check(self.lib.lrcn_train_step_staged(self._h, slot, pdrop, seed, C.byref(out)))
            return float(out.value)
        check(self.lib.lrcn_train_step_staged(self._h, slot, pdrop, seed, None))
        return None

    # ---- generation
    def beam_search(self, split, image_ids, beam_width, nword, want_logps=True):
        ids = np.ascontiguousarray(image_ids, dtype=np.int64)
        n = len(ids)
        toks = np.zeros((n, nword + 2), dtype=np.int64)
        lens = np.zeros(n, dtype=np.int32)
        prob = np.zeros(n, dtype=np.float32)
        lps = np.zeros((n, nword + 1), dtype=np.float32) if want_logps else None
        check(self.lib.lrcn_beam_search(self._h, split, _i64(ids), n, beam_width, nword, _i64(toks),
                                        lens.ctypes.data_as(_i32p), _f32(prob), _f32(lps) if want_logps else None))
        return toks, lens, prob, lps

    # ---- fc7 producer (f-4): VGG-16 up to relu7
    def set_cnn_param(self, layer, which, a):
        """layer 1..15 (conv1_1..conv5_3, fc6, fc7); which 0: filter kh x kw x Cin x Cout, 1: bias of Cout values."""
        a = np.asfortranarray(a, dtype=np.float32)
        dims = cnn_dims(layer, which)
        if a.size != int(np.prod(dims)) or (which == 0 and a.shape != dims):
            raise ValueError(f"CNN layer {layer} {'bias' if which else 'filter'}: shape {a.shape}, expected {dims}")
        check(self.lib.lrcn_set_cnn_param(self._h, layer, which, _f32(a), _i64(np.array(dims, dtype=np.int64))))

    def get_cnn_param(self, layer, which):
        dims = cnn_dims(layer, which)
        out = np.empty(dims if which == 0 else (dims[0],), dtype=np.float32, order="F")
        check(self.lib.lrcn_get_cnn_param(self._h, layer, which, _f32(out), _i64(np.array(dims, dtype=np.int64))))
        return out

    def extract_features(self, images, flags=0):
        """images: 224 x 224 x 3 x n (column-major element order) -> relu7 as an n x 4096 array (row i = image i)."""
        images = np.asfortranarray(images, dtype=np.float32)
        if images.ndim != 4 or images.shape[:3] != (CNN_IMAGE, CNN_IMAGE, 3):
            raise ValueError(f"images must be {CNN_IMAGE} x {CNN_IMAGE} x 3 x n, got {images.shape}")
        n = images.shape[3]
        out = np.zeros((n, 4096), dtype=np.float32)
        check(self.lib.lrcn_extract_features(self._h, _f32(images), n, flags, _f32(out)))
        return out

    def test_cnn_activation(self, layer, n):
        """Pre-ReLU output of CNN layer `layer` for the n images of the last extraction, H x W x Cout x n."""
        h = CNN_HOUT[layer - 1]
        out = np.zeros((h, h, CNN_SHAPES[layer - 1][3], n), dtype=np.float32, order="F")
        check(self.lib.lrcn_test_cnn_activation(self._h, layer, _f32(out), n))
        return out

    # ---- checkpoint sidecar (f-2)
    def checkpoint_save(self, path: str, with_adam: bool = True, aux: bytes = b""):
        check(self.lib.lrcn_checkpoint_save(self._h, path.encode(), 1 if with_adam else 0, aux if aux else None, len(aux)))

    def checkpoint_load(self, path: str):
        """Loads weights (+ Adam state if stored) into the handle; returns (had_adam, aux bytes)."""
        had, n = C.c_int32(), C.c_int64()
        # the sizes are in the header: a first pass with no aux buffer would load the weights twice, so size the buffer from the file
        size = os.path.getsize(path)
        buf = C.create_string_buffer(max(size, 1))
        check(self.lib.lrcn_checkpoint_load(self._h, path.encode(), C.byref(had), buf, size, C.byref(n)))
        return bool(had.value), buf.raw[:n.value]

    # ---- data parallel
    @staticmethod
    def comm_unique_id() -> bytes:
        buf = C.create_string_buffer(COMM_ID_BYTES)
        check(_Lib(load()).lrcn_comm_unique_id(buf))
        return buf.raw

    def comm_init(self, uid: bytes, rank: int, nranks: int):
        assert len(uid) == COMM_ID_BYTES
        check(self.lib.lrcn_comm_init(self._h, uid, rank, nranks))

    def p2p_export(self) -> bytes:
        buf = C.create_string_buffer(P2P_BLOB_BYTES)
        check(self.lib.lrcn_p2p_export(self._h, buf))
        return buf.raw

    def p2p_import(self, blobs: bytes, rank: int, nranks: int):
        assert len(blobs) == nranks * P2P_BLOB_BYTES
        check(self.lib.lrcn_p2p_import(self._h, blobs, rank, nranks))

    # ---- measurement
    def sync(self):
        check(self.lib.lrcn_sync(self._h))

    def timer_start(self):
        check(self.lib.lrcn_timer_start(self._h))

    def timer_stop(self) -> float:
        ms = C.c_float()
        check(self.lib.lrcn_timer_stop(self._h, C.byref(ms)))
        return float(ms.value)

    def kernel_launches(self) -> int:
        n = C.c_int64()
        check(self.lib.lrcn_kernel_launches(self._h, C.byref(n)))
        return int(n.value)

    def get_trace(self, steps):
        out = np.zeros((steps, 8), dtype=np.uint64)
        check(self.lib.lrcn_get_trace(self._h, out.ctypes.data_as(_p(C.c_uint64)), out.size))
        return out

    def flush_l2(self):
        check(self.lib.lrcn_flush_l2(self._h))

    def time_kernel(self, name: str, reps: int = 10):
        ms, by, fl = C.c_float(), C.c_double(), C.c_double()
        check(self.lib.lrcn_time_kernel(self._h, name.encode(), reps, C.byref(ms), C.byref(by), C.byref(fl)))
        return float(ms.value), float(by.value), float(fl.value)

    # ---- kernel-level test hooks
    def test_mma_rate(self, M, N, n_mma=512, commit_every=0, issuers=1):
        a, b = C.c_int64(), C.c_int64()
        check(self.lib.lrcn_test_mma_rate(self._h, M, N, n_mma, commit_every, issuers, C.byref(a), C.byref(b)))
        return a.value, b.value

    def test_gemm_time(self, a_kmajor, b_kmajor, M, N, K, shadow_out=False, iters=20, dbg=0):
        ms = C.c_float()
        check(self.lib.lrcn_test_gemm_time(self._h, int(a_kmajor), int(b_kmajor), M, N, K, int(shadow_out), iters, dbg, C.byref(ms)))
        return ms.value

    def test_gemm(self, precision, a_kmajor, b_kmajor, A, B, bias=None, C0=None):
        A = np.ascontiguousarray(A, dtype=np.float32)
        B = np.ascontiguousarray(B, dtype=np.float32)
        M, K = A.shape if a_kmajor else A.shape[::-1]
        N = B.shape[0] if b_kmajor else B.shape[1]
        assert (B.shape[1] if b_kmajor else B.shape[0]) == K
        out = np.zeros((M, N), dtype=np.float32) if C0 is None else np.ascontiguousarray(C0, dtype=np.float32).copy()
        b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
        check(self.lib.lrcn_test_gemm(self._h, precision, int(a_kmajor), int(b_kmajor), M, N, K, _f32(A), _f32(B),
                                      _f32(b) if b is not None else None, 0 if C0 is None else 1, _f32(out)))
        return out

    def test_beam_topk_logits(self, logits, parent_prob, K):
        logits = np.ascontiguousarray(logits, dtype=np.float32)
        parent_prob = np.ascontiguousarray(parent_prob, dtype=np.float32)
        R, V = logits.shape
        tok = np.zeros((R, K), dtype=np.int64)
        sc = np.zeros((R, K), dtype=np.float32)
        lp = np.zeros((R, K), dtype=np.float32)
        check(self.lib.lrcn_test_beam_topk_logits(self._h, _f32(logits), _f32(parent_prob), R, V, K, _i64(tok), _f32(sc), _f32(lp)))
        return tok, sc, lp

    def test_beam_select(self, probs, parent_prob, n_images, K, first_step):
        probs = np.ascontiguousarray(probs, dtype=np.float32)
        parent_prob = np.ascontiguousarray(parent_prob, dtype=np.float32)
        R, V = probs.shape
        assert R == n_images * K
        tok = np.zeros(R, dtype=np.int64)
        par = np.zeros(R, dtype=np.int32)
        sc = np.zeros(R, dtype=np.float32)
        check(self.lib.lrcn_test_beam_select(self._h, _f32(probs), _f32(parent_prob), n_images, K, V, int(first_step),
                                             _i64(tok), par.ctypes.data_as(_i32p), _f32(sc)))
        return tok.reshape(n_images, K), par.reshape(n_images, K), sc.reshape(n_images, K)
