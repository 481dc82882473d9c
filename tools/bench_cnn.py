"""Throughput of the fc7 producer (lrcn_extract_features, VGG-16 up to relu7) on one GPU; writes one JSON report.

  python tools/bench_cnn.py [--images 256] [--reps 3] [--out profiles/r03_cnn_bench.json]

For each precision: images/s with the images in host memory (numpy) and already on the device (a torch CUDA tensor whose
pointer goes straight to the C ABI), per-kernel times from torch.profiler over one separate extraction, achieved FLOP/s
of the GEMMs and bytes/s of the patch gathers computed from the layer shapes below, and -- for context -- torch's own
VGG-16 (cuDNN, fp32, TF32 off) on the same images and weights, with the relative difference of its relu7 to ours.
The card's name and power limit are read in the same run.  Random He-initialised weights: the timing does not depend on
the values."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import lrcn_b200  # noqa: E402,F401
from lrcn_b200 import abi  # noqa: E402
import vgg_oracle as V  # noqa: E402  (weights / images generators and layer table only; no fp64 run here)

CH = 16  # images per internal chunk (csrc/cnn_sm100.cu)


def layer_table():
    """Per layer: output size, Cin, Cout, k, K, padded K, input map size before pooling, whether the input is pooled."""
    rows, h = [], 224
    for l, (kh, _, cin, cout) in enumerate(abi.CNN_SHAPES, start=1):
        pool = (l - 1) in abi.CNN_POOL_AFTER
        hin = h // 2 if pool else h
        pad = 1 if l <= 13 else 0
        hout = hin + 2 * pad - kh + 1
        K = kh * kh * cin
        rows.append(dict(layer=l, hout=hout, cin=cin, cout=cout, k=kh, K=K, Kp=(K + 7) // 8 * 8, hprev=h, pool=pool))
        h = hout
    return rows


def per_image_counts():
    """Algorithmic FLOPs (2 x MAC, unpadded K) and, per image, the patch bytes the gathers write plus the unique bytes they read."""
    flops = gather_bytes = patch_bytes = 0
    for r in layer_table():
        M = r["hout"] ** 2
        flops += 2 * M * r["K"] * r["cout"]
        wbytes = M * r["Kp"] * 4  # fp32, or bf16 hi + lo: 4 bytes per element either way
        rbytes = (r["hprev"] ** 2) * r["cin"] * 4 if r["layer"] > 1 else 3 * 224 * 224 * 4
        gather_bytes += wbytes + rbytes
        patch_bytes += wbytes
    return flops, gather_bytes, patch_bytes


def card():
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip().splitlines()[0] if q.stdout.strip() else q.stderr.strip()
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def extract_ptr(h, dimg, n, dout, flags=0):
    fp = C.POINTER(C.c_float)
    abi.check(h.lib.lrcn_extract_features(h._h, C.cast(dimg.data_ptr(), fp), n, flags, C.cast(dout.data_ptr(), fp)))


def profile_kernels(h, dimg, n, dout):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        extract_ptr(h, dimg, n, dout)
        torch.cuda.synchronize()
    kern = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name
        cls = ("patch gather (conv1_1)" if "cnn_gather_image" in name else "patch gather" if "cnn_gather" in name else
               "relu7 / L1 tail" if "cnn_relu7" in name else "gemm" if "gemm" in name else "memset" if "emset" in name else
               "memcpy" if "emcpy" in name else "other: " + name[:80])
        d = kern.setdefault(cls, {"ms": 0.0, "launches": 0})
        d["ms"] += e.device_time / 1e3 if hasattr(e, "device_time") else e.cuda_time / 1e3
        d["launches"] += 1
    return kern


def torch_vgg(params):
    ws = [(torch.from_numpy(np.ascontiguousarray(np.transpose(w, (3, 2, 0, 1)))).cuda(), torch.from_numpy(b).cuda()) for w, b in params]

    def run(x):  # x: (n, 3, 224, 224)
        for l, (w, b) in enumerate(ws, start=1):
            x = F.relu(F.conv2d(x, w, b, padding=1 if l <= 13 else 0))
            if l in abi.CNN_POOL_AFTER:
                x = F.max_pool2d(x, 2, 2)
        return x.reshape(x.shape[0], -1)
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=256)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_cnn_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cnn needs a CUDA device")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n = a.images
    params = V.he_params(seed=0)
    images = V.random_images(n, seed=1)
    dimg = torch.from_numpy(images.ravel(order="F")).cuda()
    dout = torch.empty(n * 4096, device="cuda")
    report = {"card": card(), "images": n, "chunk": CH, "reps": a.reps, "weights": "He-initialised random", "precisions": {}}
    # torch reference first (fp32 cuDNN, TF32 off), batches of CH like ours
    run = torch_vgg(params)
    x = torch.from_numpy(np.ascontiguousarray(np.transpose(images, (3, 2, 0, 1)))).cuda()
    with torch.no_grad():
        run(x[:CH]); torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.reps):
            ref = torch.cat([run(x[i:i + CH]) for i in range(0, n, CH)])
        torch.cuda.synchronize()
        t_torch = (time.perf_counter() - t0) / a.reps
    ref = ref.cpu().numpy().astype(np.float64)
    report["torch_vgg16_fp32_no_tf32"] = {"images_per_s": n / t_torch, "s_per_call": t_torch}
    del x
    for prec, pname in ((abi.PREC_BF16X3, "bf16x3"), (abi.PREC_FP32, "fp32")):
        cfg = abi.default_config(embed=64, hidden1=64, hidden2=64, vocab=300, max_batch=4, max_len=8, max_gen_rows=12, precision=prec)
        with abi.Handle(cfg) as h:
            for layer, (w, b) in enumerate(params, start=1):
                h.set_cnn_param(layer, 0, w)
                h.set_cnn_param(layer, 1, b)
            r = {}
            h.extract_features(images[..., :2 * CH])  # warm-up: modules, tensor maps
            t0 = time.perf_counter()
            for _ in range(a.reps):
                feats = h.extract_features(images)
            t_host = (time.perf_counter() - t0) / a.reps
            extract_ptr(h, dimg, n, dout)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(a.reps):
                extract_ptr(h, dimg, n, dout)
            torch.cuda.synchronize()
            t_dev = (time.perf_counter() - t0) / a.reps
            dfeats = dout.view(n, 4096).cpu().numpy()
            r["host_images_per_s"] = n / t_host
            r["device_images_per_s"] = n / t_dev
            r["host_vs_device"] = t_host / t_dev
            r["relerr_host_vs_device_output"] = float(np.linalg.norm(feats - dfeats) / np.linalg.norm(dfeats))  # split-K sums: last bits
            r["relerr_vs_torch_fp32"] = float(np.linalg.norm(feats - ref) / np.linalg.norm(ref))
            pn = min(n, 4 * CH)
            kern = profile_kernels(h, dimg, pn, dout)
            flops, gbytes, pbytes = per_image_counts()
            gemm_ms = kern.get("gemm", {}).get("ms", 0.0)
            gat_ms = kern.get("patch gather", {}).get("ms", 0.0) + kern.get("patch gather (conv1_1)", {}).get("ms", 0.0)
            r["profile_images"] = pn
            r["kernels"] = kern
            r["algorithmic_gflop_per_image"] = flops / 1e9
            r["gemm_tflops_achieved"] = flops * pn / (gemm_ms * 1e-3) / 1e12 if gemm_ms else None
            r["gather_gb_per_image"] = gbytes / 1e9
            r["patch_gb_per_image"] = pbytes / 1e9
            r["gather_tb_per_s_achieved"] = gbytes * pn / (gat_ms * 1e-3) / 1e12 if gat_ms else None
            r["kernel_ms_per_image"] = sum(v["ms"] for v in kern.values()) / pn
            report["precisions"][pname] = r
            print(pname, json.dumps(r), flush=True)
    report["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(report, f, indent=1)
    print(json.dumps(report))


if __name__ == "__main__":
    main()
