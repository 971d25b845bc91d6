"""Launch the event-level attention backward a few times at the bench shape (B=8, S=2048, 16 heads, d=64): ncu target."""
import os
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "midi-model_b200"))
from midi_b200 import ops  # noqa: E402

B, S, nh, D = 8, 2048, 16, 64
g = torch.Generator(device="cuda").manual_seed(1)
qkv = torch.randn(B * S, 3 * nh * D, device="cuda", generator=g).to(torch.bfloat16)
do = torch.randn(B * S, nh * D, device="cuda", generator=g).to(torch.bfloat16)
o, lse = ops.attn_causal_fwd(qkv, B, S, nh, D, want_lse=True, impl="tc")
n = int(sys.argv[1]) if len(sys.argv) > 1 else 3
for _ in range(n):
    dqkv = ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, impl="tc")
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(10):
    ops.attn_causal_bwd(qkv, o, do, lse, B, S, nh, D, impl="tc")
e1.record()
torch.cuda.synchronize()
print("ms per backward", e0.elapsed_time(e1) / 10, float(dqkv.float().abs().mean()))
