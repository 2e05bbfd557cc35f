#!/usr/bin/env python
"""Developer probe: K1 (gfx_aggregate, fp16) time on a tiled synthetic shard; argv[1] = nodes."""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
import ginfinity_b200 as gb  # noqa: E402
from ginfinity_b200 import _native as nat  # noqa: E402
from ginfinity_b200.weights import fold, synthetic_state  # noqa: E402
from helpers import random_records  # noqa: E402

dev = torch.device("cuda:0")
lib = nat.lib
S = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
handle = nat.model_create(fold(synthetic_state(seed=7)))
want = int(sys.argv[1]) if len(sys.argv) > 1 else 603000
shard = gb.GraphBuilder().build_shard(random_records(0, 3000))
reps = max(1, want // shard.node_count)
N1 = shard.node_count
ei = np.concatenate([shard.edge_index + np.int32(r * N1) for r in range(reps)], axis=1)
et = np.tile(shard.edge_types, reps)
N, E = N1 * reps, shard.edge_count * reps
ei_d, et_d = torch.from_numpy(ei).to(dev), torch.from_numpy(et).to(dev)
row_ptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
col_src = torch.empty(E, dtype=torch.int32, device=dev)
col_type = torch.empty(E, dtype=torch.uint8, device=dev)
need = lib.gfx_csr_workspace_bytes(N, E)
ws = torch.empty(need, dtype=torch.uint8, device=dev)
nat.check(lib.gfx_csr_build(ei_d[0].data_ptr(), ei_d[1].data_ptr(), et_d.data_ptr(), N, E, 0,
                            row_ptr.data_ptr(), col_src.data_ptr(), col_type.data_ptr(),
                            ws.data_ptr(), need, S()))
h = torch.randn(N, 128, device=dev).half()
z = torch.empty_like(h)
run = lambda: nat.check(lib.gfx_aggregate(handle, 0, h.data_ptr(), row_ptr.data_ptr(),  # noqa: E731
                                          col_src.data_ptr(), col_type.data_ptr(), N, z.data_ptr(), 0, S()))
for _ in range(5):
    run()
torch.cuda.synchronize()
a, b = torch.cuda.Event(True), torch.cuda.Event(True)
a.record()
for _ in range(20):
    run()
b.record()
torch.cuda.synchronize()
t = a.elapsed_time(b) / 20 * 1e-3
alg = N * 516 + E * 5
print(f"K1 N={N} E={E}: {t * 1e3:.4f} ms  {t / N * 1e9:.4f} ns/node  "
      f"{alg / t / 1e9:.0f} GB/s algorithmic")
