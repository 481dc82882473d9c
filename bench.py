#!/usr/bin/env python
"""bench.py -- LRCN decoder hot path on B200 (contract in the task statement, tier section 4).

A "step" is one training step (forward, BPTT, [gradient exchange], Adam) of the 2-layer factored LSTM
caption decoder on one synthetic batch AT THE REFERENCE'S TRAINING SETTING pdrop = 0.4 (lrcn.jl:227).
Workload = BASELINE.json configs[1]: Flickr30k-shaped (fc7 4096-d, E=H1=H2=512, V=7731), 256 captions per
GPU per step, caption length l drawn per batch from the Flickr length histogram (all ranks share l; rows
differ per rank), data-parallel over N GPUs.

  value : whole-job tokens/s with the batches already resident in HBM (lrcn_train_step_staged), pdrop 0.4
  e2e   : the same metric through the reference-facing call lrcn_train_step with HOST buffers
          (token/id H2D and loss D2H inside the timed region), pdrop 0.4
  roofline : the TIME-DOMINANT kernel (the persistent LSTM backward sequence kernel), timed live with CUDA
          events on the library's stream; the vocab GEMM, the forward LSTM kernel and Adam are reported beside it
  --impl reference : the CPU restatement of the Knet path (oracle/, numpy+OpenBLAS, all host threads) on the
          same full-size batches (Julia/Knet cannot run in this image: see DESIGN.md)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (E, H1, H2, V, B per GPU, length shape)
    "flickr30k_train_b256": dict(E=512, H1=512, H2=512, V=7731, B=256, shape="flickr"),
    "flickr8k_train_b64": dict(E=512, H1=512, H2=512, V=8000, B=64, shape="fixed20"),       # configs[0], Knet-CPU case
    "coco_2f_train_b256": dict(E=1000, H1=1000, H2=1000, V=10636, B=256, shape="coco"),     # configs[3]
}
N_IMG = 8192
N_SLOTS = 16
KSLOT = N_SLOTS          # extra staged batch of fixed length for the single-kernel timings (matches the ncu captures)
KSLOT_L = {"flickr": 12, "fixed20": 20, "coco": 10}
PDROP = 0.4              # lrcn.jl:227: the reference trains at pdrop = 0.4 and nowhere else


def flops_per_token(w):
    E, H1, H2, V = w["E"], w["H1"], w["H2"], w["V"]
    C = H2 // 2
    return 6.0 * ((E + H1) * 4 * H1 + H1 * C + 2 * H2 * 4 * H2 + H2 * V)  # SURVEY §8(d): 6*M_tok


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the run (B200_PROFILING.md recipe).  Started before the warm-up; the
    report uses the samples inside the timed window and, when the window is shorter than the sampling period, the samples
    of the whole GPU-busy part of the bench (warm-up .. end-to-end run), saying which."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu"

    def __init__(self, gpu_index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(gpu_index),
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def _collect(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1:
                continue
            f = [x.strip() for x in line.split(",")]
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except Exception:
                continue
            for nm, val in zip(names, f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return sm, mx, reasons

    def stop(self, timed, busy):
        if not self.proc:
            return None
        time.sleep(0.1)
        self.proc.terminate()
        sm, mx, reasons = self._collect(timed[0] - 0.01, timed[1] + 0.03)
        window = "timed region"
        if len(sm) < 3:
            sm, mx, reasons = self._collect(busy[0], busy[1])
            window = "warm-up .. end-to-end run (the timed region is shorter than the sampling period)"
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm), "window": window}


def make_batches(w, rank, n_slots, seed=0):
    from lrcn_b200 import synth
    ls = synth.lengths(n_slots, w["shape"], seed=4 + seed)             # same on every rank
    out = []
    for s in range(n_slots):
        l = int(ls[s])
        tok = synth.tokens(l, w["B"], w["V"], seed=3 + 1000 * s + 77 * rank, zipf=True)
        img = synth.image_ids(w["B"], N_IMG, seed=5 + 1000 * s + 77 * rank)
        out.append((img, tok, l))
    return out


def oracle_masks(O, w, l, B, seed):
    return O.dropout_masks(PDROP, seed, l + 1, B, w["E"], w["H2"])


DUMP_BUDGET = 64 << 20   # bytes written by --dump-outputs at most
DUMP_SAMPLE = 1 << 20    # elements kept of a larger array


def last_step_outputs(h, B, l):
    """What the last lrcn_train_step_staged left for its caller: the nine updated weights (weight_k = parameter k of the ABI)
    and the per-token target log-probs of its forward pass [l+1][B]; `loss` is their negated mean, the value the call returns
    when asked for it.  Partial sums land in any order, and every step before this one (graph capture, warm-up, timed steps)
    trains the same weights, so two runs of one build drift apart with the step count.  Measured on a B200 at 1000 W
    (flickr30k_train_b256), two runs agreed to relative 5e-4 in every weight and 1e-5 in the loss at --steps 10, and to 2e-2
    and 2e-5 at --steps 100; the gradients are not written, as those of layer 2 drifted by 18 % at --steps 7."""
    out = {f"weight_{k}": h.get_param(k) for k in range(1, 10)}
    lp = h.token_logps(l, B)
    out["token_logps"] = lp
    out["loss"] = np.float64(-lp.sum(dtype=np.float64) / lp.size)
    return out


def dump_outputs(out_dir, arrays):
    """Writes out_dir/<name>.npy.  An array of more than DUMP_SAMPLE elements is replaced by DUMP_SAMPLE of its entries at
    sorted column-major positions drawn with a fixed seed, so that two runs or two builds compare entry for entry."""
    small = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        if a.size > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            a = a.ravel(order="F")[pos]
        small[name] = a
    assert sum(a.nbytes for a in small.values()) <= DUMP_BUDGET, f"--dump-outputs would write more than {DUMP_BUDGET} bytes"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in small.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def cpu_beam_leg(budget_s=12.0, n_max=64, K=3, nword=30):
    """BASELINE metric "beam-3 captions/s ... vs Knet CPU": the oracle's generate() (lrcn.jl:585-678 restated, host
    sortperm over V per beam per step exactly like lrcn.jl:655,667) on the COCO-shaped model, bounded sample."""
    from lrcn_b200 import synth
    from oracle import lrcn_oracle as O
    E = H = 512
    V = 10000
    model = synth.eos_timed_model([H, H], V, E)
    feats = synth.features(n_max, seed=6) * np.float32(100)
    O.generate(model, feats[0], nword, K)
    t0 = time.perf_counter()
    n, steps = 0, 0
    while n < n_max and time.perf_counter() - t0 < budget_s:
        toks, _ = O.generate(model, feats[n], nword, K)
        steps += len(toks) - 1
        n += 1
    dt = time.perf_counter() - t0
    return {"metric": f"beam-{K} captions/s", "value": n / dt, "unit": "captions/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"{n} images, beam {K}, V={V}, E=H={H}, eos-timed synthetic model (mean {steps / max(n, 1):.1f} decode steps), oracle generate()"}


def run_reference(args, w, rank, world):
    """CPU restatement of the Knet path (oracle/), numpy + OpenBLAS on all host threads: the SAME full-size batches
    (B rows, same lengths, same model, pdrop 0.4 with explicit masks), so same_config holds."""
    if rank != 0:
        return
    from lrcn_b200 import synth
    from oracle import lrcn_oracle as O
    cores = os.cpu_count() or 1
    rows = w["B"]
    model = synth.initweights([w["H1"], w["H2"]], w["V"], w["E"], seed=1)
    opt = O.initparams(model)
    feats = synth.features(256, seed=2)
    batches = make_batches(w, 0, N_SLOTS)

    def step(i):
        img, tok, l = batches[i % N_SLOTS]
        X = feats[(img - 1) % 256]
        g, _ = O.lossgradient(model, O.initstate(model, rows), X, list(tok), range(0, l), masks=oracle_masks(O, w, l, rows, 1000 + i))
        O.update(model, g, opt)
        return rows * (l + 1)

    for i in range(args.warmup):
        step(i)
    t0 = time.perf_counter()
    ntok = 0
    for i in range(args.steps):
        ntok += step(args.warmup + i)
    dt = time.perf_counter() - t0
    val = ntok / dt
    sample = f"{args.steps} full train steps (forward, BPTT, Adam; pdrop {PDROP}) on the workload's own {rows}-row batches"
    line = {"impl": "reference", "metric": "train tokens/s", "value": val, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, **{k: w[k] for k in ("E", "H1", "H2", "V")}, "batch_per_gpu": w["B"], "global_batch": w["B"],
                       "lengths": w["shape"], "pdrop": PDROP},
            "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU restatement of lrcn.jl's Knet path (Julia/Knet not installable in this image); one process on all host cores"}
    if not args.no_beam:
        line["beam"] = cpu_beam_leg()
    print(json.dumps(line), flush=True)


def cpu_baseline_leg(w):
    """Bounded oracle sample on the host cores (rank 0, N=1): ~10-30 s of CPU work on the workload's own batches."""
    from lrcn_b200 import synth
    from oracle import lrcn_oracle as O
    rows = w["B"]
    model = synth.initweights([w["H1"], w["H2"]], w["V"], w["E"], seed=1)
    opt = O.initparams(model)
    feats = synth.features(256, seed=2)
    batches = make_batches(w, 0, 4)

    def step(i):
        img, tok, l = batches[i % 4]
        g, _ = O.lossgradient(model, O.initstate(model, rows), feats[(img - 1) % 256], list(tok), range(0, l), masks=oracle_masks(O, w, l, rows, i))
        O.update(model, g, opt)
        return rows * (l + 1)

    t0 = time.perf_counter()
    ntok, n = 0, 0
    while time.perf_counter() - t0 < 15.0 and n < 6:
        ntok += step(n)
        n += 1
    dt = time.perf_counter() - t0
    return {"value": ntok / dt, "unit": "tokens/s", "cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"{n} oracle train steps (numpy/OpenBLAS fp32, pdrop {PDROP}) on the workload's own {rows}-row batches"}


def beam_leg(local_rank, rank, world, prec, max_over_ranks, barrier, shaped, n_img=1024, K=3, nword=30):
    """BASELINE.json configs[2]: COCO-shaped beam-search generation (E=H=512, V=10000, beam 3, nword 30), images sharded
    across ranks with no collective.  shaped=True: synth.eos_timed_model, decodes end after an image-dependent number of
    steps (mean ~11, like COCO captions, SURVEY §8d).  shaped=False: random weights never emit eos, every image decodes
    the full nword+1 = 31 steps (the WORST case).  `row_steps_per_s` (beam rows advanced one step per second) is the
    length-independent figure.  Host ids in, host tokens out (e2e by construction); wall clock, max over ranks."""
    from lrcn_b200 import abi, synth
    E = H = 512
    V = 10000
    cfg = abi.default_config(embed=E, hidden1=H, hidden2=H, vocab=V, max_batch=8, max_len=2, max_gen_rows=n_img * K, device=local_rank,
                             precision=prec, use_graphs=0)
    with abi.Handle(cfg) as g:
        g.set_model(synth.eos_timed_model([H, H], V, E) if shaped else synth.initweights([H, H], V, E, seed=1))
        ids = np.arange(1, n_img + 1, dtype=np.int64) + 100000 * rank
        g.load_features(1, ids, synth.features(n_img, seed=6 + rank) * np.float32(100 if shaped else 1))
        g.beam_search(1, ids, K, nword, want_logps=False)  # warm-up
        barrier()
        t0 = time.perf_counter()
        reps = 3
        steps = 0
        for _ in range(reps):
            toks, lens, prob, _ = g.beam_search(1, ids, K, nword, want_logps=False)
            steps += int(lens.max()) - 1
        g.sync()
        dt = max_over_ranks(time.perf_counter() - t0)
    rowsteps = float((lens - 1).sum()) * K  # rows that had to be advanced if finished images stopped costing anything
    return {"metric": f"beam-{K} captions/s", "value": reps * n_img * world / dt, "unit": "captions/s", "images_per_gpu": n_img, "beam_width": K,
            "nword": nword, "vocab": V, "mean_decode_steps": float(lens.mean() - 1), "max_decode_steps": steps / reps, "ms_per_batch": 1e3 * dt / reps,
            "row_steps_per_s": n_img * K * (steps / reps) * world / (dt / reps), "useful_row_steps_per_s": rowsteps * world / (dt / reps),
            "model": "eos-timed synthetic model (COCO-shaped decode lengths)" if shaped else "random weights: eos never wins, full 31 steps (worst case)",
            "timing": "wall clock around lrcn_beam_search (host ids in, host tokens out), max over ranks"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="flickr30k_train_b256", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-beam", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (updated weights, token log-probs, loss) "
                         "as DIR/<name>.npy; arrays of more than 2^20 elements as a fixed seeded sample")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3)
    w = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import lrcn_b200  # noqa: F401
    if args.impl == "reference":
        run_reference(args, w, rank, world)
        return

    from lrcn_b200 import abi, synth
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sampler = ClockSampler(local_rank) if rank == 0 else None  # before any GPU work: the line's `clocks` is never null
    prec = abi.PREC_BF16X3 if args.precision == "bf16x3" else abi.PREC_FP32
    cfg = abi.default_config(embed=w["E"], hidden1=w["H1"], hidden2=w["H2"], vocab=w["V"], max_batch=w["B"], max_len=28,
                             max_gen_rows=8, device=local_rank, precision=prec, use_graphs=1)
    h = abi.Handle(cfg)
    h.set_model(synth.initweights([w["H1"], w["H2"]], w["V"], w["E"], seed=1))
    h.load_features(0, np.arange(1, N_IMG + 1, dtype=np.int64), synth.features(N_IMG, seed=2))
    dp_exchange = None
    if world > 1:
        import torch
        uid = torch.zeros(abi.COMM_ID_BYTES, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid = torch.frombuffer(bytearray(abi.Handle.comm_unique_id()), dtype=torch.uint8).cuda()
        dist.broadcast(uid, 0)
        h.comm_init(bytes(uid.cpu().numpy().tobytes()), rank, world)
        # peer-memory gradient exchange (csrc/dp_p2p.cu): every rank exports its IPC blob, all-gather, import
        mine = torch.frombuffer(bytearray(h.p2p_export()), dtype=torch.uint8).cuda()
        blobs = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(blobs, mine)
        ok = 1
        try:
            h.p2p_import(b"".join(bytes(b.cpu().numpy().tobytes()) for b in blobs), rank, world)
        except abi.LrcnError as e:  # no peer access between these GPUs
            ok = 0
            print(f"[bench] rank {rank}: peer memory unavailable ({e})", file=sys.stderr)
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)  # the choice must be the same on every rank
        if int(flag.item()) == 0:
            os.environ["LRCN_DP_NCCL"] = "1"  # read by the library at the first data-parallel step
        dp_exchange = "nccl" if os.environ.get("LRCN_DP_NCCL") else "p2p"

    batches = make_batches(w, rank, N_SLOTS)
    for s, (img, tok, l) in enumerate(batches):
        h.stage_batch(s, 0, img, tok)
    kl = KSLOT_L[w["shape"]]
    h.stage_batch(KSLOT, 0, synth.image_ids(w["B"], N_IMG, seed=991 + rank), synth.tokens(kl, w["B"], w["V"], seed=992 + rank, zipf=True))

    def barrier():
        h.sync()
        if dist is not None:
            dist.barrier()
            import torch
            torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- setup: capture the CUDA graph of every step shape (one per distinct caption length and dropout on/off) before
    # anything is timed: graph capture + instantiation is this framework's "compile" step and costs milliseconds per shape
    seen = set()
    for s_, (_, _, l_) in enumerate(batches):
        if l_ not in seen:
            seen.add(l_)
            h.train_step_staged(s_, PDROP, 7)
            h.train_step_staged(s_, 0.0, 7)
    h.train_step_staged(KSLOT, PDROP, 7)
    h.sync()
    barrier()
    t_busy0 = time.time()

    def timed_run(pdrop, seed0):
        for i in range(args.warmup):
            h.train_step_staged(i % N_SLOTS, pdrop, seed0 + i)
        barrier()
        launches0 = h.kernel_launches()
        t0 = time.time()
        h.timer_start()
        ntok = 0
        for i in range(args.steps):
            s = (args.warmup + i) % N_SLOTS
            h.train_step_staged(s, pdrop, seed0 + 1000 + i)
            ntok += w["B"] * (batches[s][2] + 1)
        ms = h.timer_stop()
        barrier()
        t1 = time.time()
        return max_over_ranks(ms), ntok, h.kernel_launches() - launches0, (t0, t1)

    # ---- device-resident run at the reference's training setting: `value`
    ms, ntok, launches, t_timed = timed_run(PDROP, 0)
    value = ntok * world / (ms * 1e-3)
    outputs = None
    if args.dump_outputs:  # read now: the runs below train the same weights further
        if rank == 0:
            outputs = last_step_outputs(h, w["B"], batches[(args.warmup + args.steps - 1) % N_SLOTS][2])
        barrier()  # no peer starts the next exchange into this rank's buffers while they are read
    # ---- the same with dropout off (what round 1 timed), reported beside it
    ms0, ntok0, _, _ = timed_run(0.0, 5000)

    # ---- end-to-end run through the reference-facing call with host buffers: `e2e`
    for i in range(3):
        h.train_step(0, batches[i][0], batches[i][1], PDROP, i)
    barrier()
    h.timer_start()
    ntok_e = 0
    h2d = d2h = 0
    for i in range(args.steps):
        img, tok, l = batches[(args.warmup + i) % N_SLOTS]
        h.train_step(0, img, tok, PDROP, 2000 + i)          # H2D of tokens/ids/scalars and D2H of the loss inside
        ntok_e += w["B"] * (l + 1)
        h2d += (2 * (l + 1) * w["B"] + w["B"]) * 4 + 64
        d2h += 8
    ms_e = max_over_ranks(h.timer_stop())
    barrier()
    e2e_val = ntok_e * world / (ms_e * 1e-3)
    # ---- the same steps through ONE lrcn_train_epoch call (SURVEY 8 row f-1): host token matrix / image ids / batch order in,
    # per-step losses out; the epoch's upload, the device-side id lookup and batch staging and the final D2H are all timed
    ep_seq = np.concatenate([b[1] for b in batches]).astype(np.int64)
    ep_ids = np.stack([b[0] for b in batches]).astype(np.int64)
    ep_len = np.array([b[2] for b in batches], dtype=np.int64)
    ep_order = np.array([(args.warmup + i) % N_SLOTS for i in range(args.steps)], dtype=np.int64)
    h.train_epoch(0, ep_seq, ep_ids, ep_len, ep_order[:3], PDROP, 3000)
    barrier()
    h.timer_start()
    ep_losses = h.train_epoch(0, ep_seq, ep_ids, ep_len, ep_order, PDROP, 4000)
    ms_ep = max_over_ranks(h.timer_stop())
    barrier()
    assert len(ep_losses) == args.steps and all(np.isfinite(ep_losses))
    e2e_epoch = {"value": ntok_e * world / (ms_ep * 1e-3), "unit": "tokens/s", "ms_per_step": ms_ep / args.steps,
                 "h2d_bytes_per_epoch": int(ep_seq.nbytes + ep_ids.nbytes) + 64 * args.steps, "d2h_bytes_per_epoch": 8 * args.steps + 8,
                 "note": "one lrcn_train_epoch call for all timed steps: host buffers in, per-step losses out, batches staged on the device"}
    t_busy1 = time.time()
    clocks = sampler.stop(t_timed, (t_busy0, t_busy1)) if sampler else None

    # ---- secondary metric of BASELINE.json: beam-3 captions/s (COCO-shaped generation, images sharded by rank, no collective)
    beam = beam_worst = None
    if not args.no_beam:
        beam = beam_leg(local_rank, rank, world, prec, max_over_ranks, barrier, shaped=True)
        beam_worst = beam_leg(local_rank, rank, world, prec, max_over_ranks, barrier, shaped=False)

    # leave valid activations/gradients of the fixed-length slot in the buffers for the single-kernel timings below
    # (collective: every rank steps)
    h.train_step_staged(KSLOT, PDROP, 1)
    barrier()

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops", 1590.0)
        peak_tf_sus = peaks.get("bf16_tflops_sustained", peak_tf)
        peak_bw = peaks.get("hbm_gbs", 6650.0)
        src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
        ncu = {}
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json"))).get(args.workload, {})
        except Exception:
            pass

        def tensor_roof(kname, label, note, reps=10, peak=peak_tf, peak_kind="burst"):
            k_ms, k_bytes, k_flops = h.time_kernel(kname, reps)
            n = ncu.get(kname, {}) if prec else {}
            same_shape = n.get("l") == kl
            return {"bound": "tensor", "kernel": label, "achieved": k_flops / (k_ms * 1e-3) / 1e12, "peak": peak, "unit": "TFLOP/s",
                    "frac": k_flops / (k_ms * 1e-3) / 1e12 / peak, "traffic": n.get("traffic_bytes") if same_shape else None,
                    "peak_source": f"{src}, {peak_kind}", "algorithmic_flops": k_flops, "launch_ms": k_ms, "shape": {"B": w["B"], "l": kl, "T": kl + 1},
                    "tensor_pipe_pct_of_elapsed_ncu": n.get("tensor_pipe_pct_of_elapsed") if same_shape else None,
                    "tensor_pipe_pct_of_active_ncu": n.get("tensor_pipe_pct_of_active") if same_shape else None, "note": note}

        lat_note = ("latency-bound persistent kernel: T-1 dependent recurrent steps, each a grid barrier + TMA of the new tile + MMA chain + cell "
                    "epilogue; achieved counts ALGORITHMIC flops 2*B*4H*H per step (the bf16x3 split issues 3x that)")
        roof = tensor_roof("lstm_bwd", "lstm_bwd_seq (layer-2 BPTT, all T steps in one launch: recurrent GEMM dG*Wh' fused with the cell adjoint)", lat_note)
        roof["share_of_step_ncu"] = ncu.get("lstm_bwd", {}).get("share_of_step") if prec else None
        roof_fwd = tensor_roof("lstm_fwd", "lstm_fwd_seq (layer-2 forward, all T steps in one launch: recurrent GEMM h*Wh fused with the LSTM cell)", lat_note)
        roof_vocab = tensor_roof("vocab_gemm", "gemm2_bf16x3_kernel<K,K> (vocab projection h2*Wout+bout: 2-CTA 256x256 tcgen05, 3 split passes)" if prec else "sgemm_kernel",
                                 "achieved counts ALGORITHMIC flops (2MNK); the bf16x3 split issues 3x that on the tensor pipe, so the ceiling of frac is 1/3; "
                                 "L2 flushed between the timed launches")
        a_ms, a_bytes, _ = h.time_kernel("adam", 10)
        roof_adam = {"bound": "hbm", "kernel": "adam_kernel", "achieved": a_bytes / (a_ms * 1e-3) / 1e9, "peak": peak_bw, "unit": "GB/s",
                     "frac": a_bytes / (a_ms * 1e-3) / 1e9 / peak_bw, "traffic": ncu.get("adam", {}).get("traffic_bytes") if prec else None,
                     "algorithmic_bytes": a_bytes, "launch_ms": a_ms, "peak_source": src}
        g_ms, g_bytes, _ = h.time_kernel("gather", 10)
        roof_gather = {"bound": "hbm", "kernel": "gather_embed_kernel (K1: vectorised word-embedding gather + bf16 hi/lo split)", "achieved": g_bytes / (g_ms * 1e-3) / 1e9,
                       "peak": peak_bw, "unit": "GB/s", "frac": g_bytes / (g_ms * 1e-3) / 1e9 / peak_bw, "algorithmic_bytes": g_bytes, "launch_ms": g_ms,
                       "traffic": None, "peak_source": src, "note": "small kernel (tens of MB): launch + tail dominated"}
        step_flops = flops_per_token(w) * ntok / args.steps
        step_tf = step_flops / (ms / args.steps * 1e-3) / 1e12
        line = {"metric": "train tokens/s", "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16x3 (bf16 hi/lo split on tcgen05, fp32 accumulate; fp32-equivalent)" if prec else "f32", "data": "synthetic",
                "config": {"workload": args.workload, **{k: w[k] for k in ("E", "H1", "H2", "V")}, "batch_per_gpu": w["B"],
                           "global_batch": w["B"] * world, "lengths": w["shape"], "pdrop": PDROP,
                           "parallelism": f"dp{world}" + (f" ({dp_exchange} gradient exchange)" if dp_exchange else ""),
                           "l2": "per-step working set (params+grads+Adam 4x53 MB, logits ~100 MB) exceeds the 126 MB L2; no explicit flush"},
                "e2e": {"value": e2e_val, "unit": "tokens/s", "h2d_bytes_per_step": h2d // args.steps, "d2h_bytes_per_step": d2h // args.steps,
                        "ms_per_step": ms_e / args.steps},
                "e2e_epoch": e2e_epoch,
                "value_pdrop0": {"value": ntok0 * world / (ms0 * 1e-3), "ms_per_step": ms0 / args.steps, "note": "same steps with dropout off (the round-1 setting)"},
                "gpu_launches": launches, "clocks": clocks,
                "step_tflops_algorithmic": step_tf, "step_frac_of_peak": {"burst": step_tf / peak_tf, "sustained": step_tf / peak_tf_sus},
                "roofline": roof, "roofline_lstm_fwd": roof_fwd, "roofline_vocab": roof_vocab, "roofline_adam": roof_adam, "roofline_gather": roof_gather}
        if beam is not None:
            line["beam"] = beam
            line["beam_worst_case"] = beam_worst
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_leg(w)
            if not args.no_beam:
                line["cpu_baseline_beam"] = cpu_beam_leg()
    if dist is not None:
        dist.barrier()  # nobody unmaps its arenas while a peer may still be inside an exchange kernel
    h.close()
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    if line is not None:
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
