"""One launch each of the score kernels at a benchmark shape (for ncu): S2 kind::i8 (tensor cores), S1 table."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from epilogos_b200 import engine, synth  # noqa: E402

bins = int(sys.argv[1]) if len(sys.argv) > 1 else 15_500_000
cols = int(sys.argv[2]) if len(sys.argv) > 2 else 833
k = int(sys.argv[3]) if len(sys.argv) > 3 else 18
x = synth.synth_states_device(bins, cols, k, seed=1)
cnt = engine.bin_counts(x, cols, k)
del x
out = torch.empty((bins, k), dtype=torch.float32, device="cuda")
n1, n2 = engine.expected_tables(cnt, cols)
e1, e2 = engine.normalize(n1), engine.normalize(n2)
for _ in range(2):
    engine.scores_s2(cnt, cols, e2, out32=out)
    engine.scores_s1(cnt, cols, e1, out32=out)
torch.cuda.synchronize()
print("done")
