"""Cost of per-tensor gradient clipping (lrcn_set_gclip) on the training step.

flickr30k_train_b256 (E = H = 512, V = 7731, B = 256, Flickr-shaped caption lengths), bf16x3, pdrop 0.4, through
lrcn_train_step_staged (the call bench.py times).  Three settings, alternated within each round:
  off   gclip = 0 (the reference; no norm launch is enqueued)
  inert gclip = 1e30 (the norm launches run, nothing is clipped)
  half  gclip = the median of the nine gradient norms of a probe step (about half of the tensors are clipped)
plus one round of the three at coco_2f_train_b256 (E = H = 1000, C = 500, V = 10636, B = 256).  Records the card's name and power
limit beside the numbers, ms per step (CUDA events on the library's stream) and kernel launches per step.

    python tools/bench_gclip.py [--steps 200] [--rounds 3] [--out profiles/r03_gclip_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import lrcn_b200  # noqa: E402,F401
from lrcn_b200 import abi, synth  # noqa: E402

WORKLOADS = {
    "flickr30k_train_b256": dict(E=512, H=512, V=7731, B=256, shape="flickr"),
    "coco_2f_train_b256": dict(E=1000, H=1000, V=10636, B=256, shape="coco"),
}
N_IMG, N_SLOTS, PDROP = 8192, 16, 0.4


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clk = [x.strip() for x in q.stdout.strip().split("\n")[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clk}


def setup(w):
    cfg = abi.default_config(embed=w["E"], hidden1=w["H"], hidden2=w["H"], vocab=w["V"], max_batch=w["B"], max_len=28, max_gen_rows=8,
                             precision=abi.PREC_BF16X3, use_graphs=1)
    h = abi.Handle(cfg)
    h.set_model(synth.initweights([w["H"], w["H"]], w["V"], w["E"], seed=1))
    h.load_features(0, np.arange(1, N_IMG + 1, dtype=np.int64), synth.features(N_IMG, seed=2))
    ls = synth.lengths(N_SLOTS, w["shape"], seed=4)
    for s in range(N_SLOTS):
        h.stage_batch(s, 0, synth.image_ids(w["B"], N_IMG, seed=5 + 1000 * s), synth.tokens(int(ls[s]), w["B"], w["V"], seed=3 + 1000 * s, zipf=True))
    img, tok = synth.image_ids(w["B"], N_IMG, seed=5), synth.tokens(int(ls[0]), w["B"], w["V"], seed=3, zipf=True)
    h.grad(0, img, tok, PDROP, 1)
    norms = h.grad_norms()
    settings = {"off": 0.0, "inert": 1e30, "half": float(np.sort(norms)[4])}
    for g in settings.values():  # capture every (length, clip on/off) graph before anything is timed
        h.set_gclip(g)
        for s in range(N_SLOTS):
            h.train_step_staged(s, PDROP, 7)
    h.sync()
    return h, settings, norms


def timed(h, gclip, steps, warmup, seed0):
    h.set_gclip(gclip)
    for i in range(warmup):
        h.train_step_staged(i % N_SLOTS, PDROP, seed0 + i)
    h.sync()
    n0 = h.kernel_launches()
    h.timer_start()
    for i in range(steps):
        h.train_step_staged((warmup + i) % N_SLOTS, PDROP, seed0 + 1000 + i)
    ms = h.timer_stop()
    h.sync()
    return ms / steps, (h.kernel_launches() - n0) / steps


def run(name, rounds, steps, warmup):
    w = WORKLOADS[name]
    h, settings, norms = setup(w)
    order = list(settings)
    res = {k: {"gclip": v, "ms_per_step": [], "launches_per_step": None} for k, v in settings.items()}
    for r in range(rounds):
        for k in order[r % 3:] + order[:r % 3]:  # rotate the order between rounds
            ms, lps = timed(h, settings[k], steps, warmup, 10000 * r)
            res[k]["ms_per_step"].append(ms)
            res[k]["launches_per_step"] = lps
    h.close()
    for k in res:
        x = res[k]["ms_per_step"]
        res[k]["median_ms"] = float(np.median(x))
        res[k]["spread_ms"] = float(max(x) - min(x))
        res[k]["tensors_clipped_at_probe"] = int((norms > res[k]["gclip"]).sum()) if res[k]["gclip"] > 0 else 0
    off = res["off"]["median_ms"]
    for k in ("inert", "half"):
        res[k]["vs_off"] = res[k]["median_ms"] / off - 1.0
    return {"workload": name, "precision": "bf16x3", "pdrop": PDROP, "rounds": rounds, "steps_per_round": steps,
            "probe_grad_norms": norms.tolist(), "settings": res}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_gclip_bench.json"))
    args = ap.parse_args()
    out = {"card": card(), "timing": "CUDA events on the library's stream around `steps` lrcn_train_step_staged calls",
           "runs": [run("flickr30k_train_b256", args.rounds, args.steps, args.warmup),
                    run("coco_2f_train_b256", 1, args.steps, args.warmup)]}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for r in out["runs"]:
        print(r["workload"], {k: (round(v["median_ms"], 4), round(v["spread_ms"], 4), v["launches_per_step"]) for k, v in r["settings"].items()})


if __name__ == "__main__":
    main()
