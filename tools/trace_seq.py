"""Per-step timeline of the persistent forward LSTM kernel (CTA (0,0), layer 2): where the step-to-step latency goes."""
import os
import sys

import numpy as np

os.environ["LRCN_SEQ_TRACE"] = "1"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lrcn_b200  # noqa: E402,F401
from lrcn_b200 import abi, synth  # noqa: E402
import bench  # noqa: E402

w = bench.WORKLOADS["flickr30k_train_b256"]
cfg = abi.default_config(embed=w["E"], hidden1=w["H1"], hidden2=w["H2"], vocab=w["V"], max_batch=w["B"], max_len=28, max_gen_rows=8,
                         precision=abi.PREC_BF16X3, use_graphs=1)
h = abi.Handle(cfg)
h.set_model(synth.initweights([w["H1"], w["H2"]], w["V"], w["E"], seed=1))
h.load_features(0, np.arange(1, 1025, dtype=np.int64), synth.features(1024, seed=2))
l = 12
h.stage_batch(0, 0, synth.image_ids(w["B"], 1024), synth.tokens(l, w["B"], w["V"], zipf=True))
for i in range(4):
    h.train_step_staged(0, 0.0, i)
h.sync()
T = l + 1
# seq4: [T][4 chains][8]: 0 barrier open (producer) | 1 chunk's TMAs issued | 2 kb0 landed (issuer) | 3 last kb landed | 4 tfull committed |
#                         5 epilogue saw tfull | 6 team done (cells, h stored) | 7 release done
tr = h.get_trace(T).astype(np.int64)
if os.environ.get("LRCN_TRACE_BWD"):
    print("BACKWARD kernel. ns relative to chain 0's barrier-open of the step; per chain: open, tma_issued, kb0, kbLast, tfull_commit, epi_start, sent, received")
    for t in range(T - 2, -1, -1):
        base = tr[t, 0, 0]
        for c in range(2):
            print(f"t={t:2d} c={c}", [int(x - base) if x else -1 for x in tr[t, c]])
        if t > 0:
            print("      next step's chain-0 barrier opens at", int(tr[t - 1, 0, 0] - base))
    h.close()
    sys.exit(0)
print("ns relative to chain 0's barrier-open of the step; per chain: open, tma_issued, kb0, kbLast, tfull_commit, epi_start, team_done, released")
for t in range(1, T):
    base = tr[t, 0, 0]
    for c in range(4):
        print(f"t={t:2d} c={c}", [int(x - base) if x else -1 for x in tr[t, c]])
    if t + 1 < T:
        print("      next step's chain-0 barrier opens at", int(tr[t + 1, 0, 0] - base))
h.close()
