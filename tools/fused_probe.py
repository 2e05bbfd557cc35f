#!/usr/bin/env python
"""Developer probe: run a fused layer entry point (argv[1]: gfx_layer_fused_pair or
gfx_layer_fused_banded, default the pair kernel) a few times on a synthetic
graph, for ncu captures."""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from ginfinity_b200 import _native as nat  # noqa: E402
from ginfinity_b200.weights import fold, synthetic_state  # noqa: E402
import ginfinity_b200 as gb  # noqa: E402
from helpers import random_records  # noqa: E402

dev = torch.device("cuda:0")
lib = nat.lib
S = lambda: torch.cuda.current_stream().cuda_stream  # noqa: E731
handle = nat.model_create(fold(synthetic_state(seed=7)))
shard = gb.GraphBuilder().build_shard(random_records(0, 3000))
N, E = shard.node_count, shard.edge_count
ei, et = torch.from_numpy(shard.edge_index).to(dev), torch.from_numpy(shard.edge_types).to(dev)
row_ptr = torch.empty(N + 1, dtype=torch.int32, device=dev)
col_src = torch.empty(E, dtype=torch.int32, device=dev)
col_type = torch.empty(E, dtype=torch.uint8, device=dev)
need = lib.gfx_csr_workspace_bytes(N, E)
ws = torch.empty(need, dtype=torch.uint8, device=dev)
nat.check(lib.gfx_csr_build(ei[0].data_ptr(), ei[1].data_ptr(), et.data_ptr(), N, E, 0,
                            row_ptr.data_ptr(), col_src.data_ptr(), col_type.data_ptr(),
                            ws.data_ptr(), need, S()))
h = torch.randn(N, 128, device=dev).half()
out = torch.empty_like(h)
name = sys.argv[1] if len(sys.argv) > 1 else "gfx_layer_fused_pair"
entry = getattr(lib, name)
desc = torch.empty(N, dtype=torch.int32, device=dev)
nat.check(lib.gfx_row_describe(row_ptr.data_ptr(), col_src.data_ptr(), col_type.data_ptr(), N,
                               desc.data_ptr(), S()))
def run():
    if name == "gfx_layer_fused_banded":
        nat.check(entry(handle, 0, h.data_ptr(), row_ptr.data_ptr(), col_src.data_ptr(),
                        col_type.data_ptr(), desc.data_ptr(), N, out.data_ptr(), S()))
    else:
        nat.check(entry(handle, 0, h.data_ptr(), row_ptr.data_ptr(), col_src.data_ptr(),
                        col_type.data_ptr(), N, out.data_ptr(), S()))
for _ in range(4):
    run()
torch.cuda.synchronize()
a, b = torch.cuda.Event(True), torch.cuda.Event(True)
a.record()
for _ in range(10):
    run()
b.record()
torch.cuda.synchronize()
print("ok", name, N, E, "fused layer %.3f ms" % (a.elapsed_time(b) / 10))
