"""Timeline of one data-parallel training step (rank 0): %globaltimer stamps placed in the step's CUDA graph (LRCN_DP_STAMPS=1).
Run under torchrun:  python -m torch.distributed.run --nproc-per-node N tools/dp_timeline.py"""
import os
import sys

import numpy as np

os.environ["LRCN_DP_STAMPS"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
import lrcn_b200  # noqa: E402,F401
from lrcn_b200 import abi, synth  # noqa: E402
import bench  # noqa: E402

rank, world, lr = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
torch.cuda.set_device(lr)
dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
w = bench.WORKLOADS["flickr30k_train_b256"]
cfg = abi.default_config(embed=w["E"], hidden1=w["H1"], hidden2=w["H2"], vocab=w["V"], max_batch=w["B"], max_len=28, max_gen_rows=8,
                         precision=abi.PREC_BF16X3, use_graphs=1, device=lr)
h = abi.Handle(cfg)
h.set_model(synth.initweights([w["H1"], w["H2"]], w["V"], w["E"], seed=1))
h.load_features(0, np.arange(1, 1025, dtype=np.int64), synth.features(1024, seed=2))
mine = torch.frombuffer(bytearray(h.p2p_export()), dtype=torch.uint8).cuda()
blobs = [torch.zeros_like(mine) for _ in range(world)]
dist.all_gather(blobs, mine)
h.p2p_import(b"".join(bytes(b.cpu().numpy().tobytes()) for b in blobs), rank, world)
l = 12
h.stage_batch(0, 0, synth.image_ids(w["B"], 1024, seed=rank), synth.tokens(l, w["B"], w["V"], zipf=True, seed=rank))
for i in range(30):
    h.train_step_staged(0, 0.4, i)
h.sync()
dist.barrier()
raw = np.zeros(64, dtype=np.uint64)
abi.check(h.lib.lrcn_get_trace(h._h, raw.ctypes.data_as(abi._p(abi.C.c_uint64)), raw.size))
t = raw.astype(np.int64)
names = {0: "step start", 1: "forward done", 2: "seg1 (vocab bwd) done", 3: "seg2 (layer-2 bwd) done", 4: "seg31 (L1 BPTT + dWemb) done", 5: "seg32 (dW1) done",
         6: "last exchange done", 7: "joined"}
for k, nm in enumerate(["bucket0 Wout", "bucket1 W2..", "bucket2 W1 (main)", "bucket3 Wemb"]):
    for j, ph in ((0, "enter"), (2, "exchange kernel done"), (3, "bf16 split done")):
        names[8 + 4 * k + j] = f"{nm}: {ph}"
if rank == 0:
    for i in sorted(names, key=lambda i: t[i]):
        if t[i]:
            print(f"{(t[i] - t[0]) / 1e3:9.1f} us  [{i:2d}] {names[i]}")
dist.barrier()
h.close()
dist.destroy_process_group()
