"""Per-phase cycle counters of the level-1 window-attention kernel (bde_tc_debug_enable + p.dbg):
total / index + LayerNorm / q,k,v GEMMs / bias table / attention / projection + scatter, averaged over the CTAs."""
import ctypes as C
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bde2vid_b200 import _lib, ops  # noqa: E402
from bde2vid_b200.engine import window_token_map  # noqa: E402

DEV = "cuda"
lib = _lib.require_device()
lib.bde_tc_debug_enable.argtypes = [C.c_size_t]
lib.bde_tc_debug_read.argtypes = [C.c_void_p, C.c_size_t]
g = torch.Generator().manual_seed(1)
# C = 64, 16 heads of 4 channels, 1976 windows (4 sequences of 132 x 176)
B, h, w, Cc, heads, D, q_ind = 4, 132, 176, 64, 16, 3, 1
P = B * h * w
tm, _ = window_token_map(B, h, w, (7, 7), False, DEV)
nwin = tm.shape[0]
frames = [(torch.randn(P, Cc, generator=g)).to(DEV) for _ in range(D)]
wqkv = (torch.randn(3 * Cc, Cc, generator=g) / 8).to(torch.bfloat16).to(DEV)
bqkv = (torch.randn(3 * Cc, generator=g) * 0.1).to(DEV)
tbl = (torch.randn(heads, D, 169, generator=g) * 0.5).to(DEV)
wproj = (torch.randn(Cc, Cc, generator=g) / 8).to(torch.bfloat16).to(DEV)
bproj = (torch.randn(Cc, generator=g) * 0.1).to(DEV)


def run64():
    xs = frames[q_ind].clone()
    fr = list(frames)
    fr[q_ind] = xs
    ops.window_attention_fused(fr, q_ind, tm.view(-1), nwin, Cc, heads, wqkv, bqkv, tbl, wproj, bproj, xs=xs)


for _ in range(3):
    run64()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10):
    run64()
e1.record()
torch.cuda.synchronize()
us = e0.elapsed_time(e1) * 100
lib.bde_tc_debug_enable(4096)
run64()
torch.cuda.synchronize()
buf = np.zeros((4096, 8), dtype=np.int64)
lib.bde_tc_debug_read(buf.ctypes.data_as(C.c_void_p), 4096)
lib.bde_tc_debug_enable(0)
used = buf[buf[:, 0] != 0]
m = used.mean(0)
print("level 1  %d windows  %.1f us (incl. the clone) | cycles per CTA (2 CTAs / SM): total %d  index+LN %d  qkv-gemm %d  tbl %d  "
      "attention %d  proj+scatter %d" % (nwin, us, m[0], m[1], m[3], m[4], m[5], m[6]))
