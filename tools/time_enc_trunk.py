"""Fused image-encoder trunk (mmf_enc_trunk) against torch conv2d in fp32: relative error, a bit-identical rerun on
the same scratch, and the CUDA-event time of one launch over n images.
Usage: python tools/time_enc_trunk.py [n_check=300] [n_time=16384] [reps=20]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from multimodalfilter_b200 import ops

torch.backends.cudnn.allow_tf32 = False
dev = torch.device("cuda:0")
torch.manual_seed(0)
n_check = int(sys.argv[1]) if len(sys.argv) > 1 else 300
n_time = int(sys.argv[2]) if len(sys.argv) > 2 else 16384
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 20
c1 = torch.nn.Conv2d(1, 32, 5, padding=2).to(dev)
c2a = torch.nn.Conv2d(32, 32, 3, padding=1).to(dev)
c2b = torch.nn.Conv2d(32, 32, 3, padding=1).to(dev)
c3 = torch.nn.Conv2d(32, 16, 3, padding=1).to(dev)
c4 = torch.nn.Conv2d(16, 8, 3, padding=1).to(dev)
w = ops.enc_pack_trunk([c1, c2a, c2b, c3, c4])
sc = ops.enc_trunk_scratch(dev)

img = torch.rand(n_check, 32, 32, device=dev) * 2 - 1
with torch.no_grad():
    x = F.relu(c1(img[:, None]))
    ref = c4(F.relu(c3(F.relu(c2b(F.relu(c2a(x))) + x))))
out = ops.enc_trunk(img, w, sc, 8)
out2 = ops.enc_trunk(img, w, sc, 8)
torch.cuda.synchronize()
print(f"{n_check} images: rel err {float((out - ref).abs().max() / ref.abs().max()):.3e}, "
      f"second run identical {bool(torch.equal(out, out2))}")

img = torch.rand(n_time, 32, 32, device=dev) * 2 - 1
for _ in range(3):
    ops.enc_trunk(img, w, sc, 8)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    ops.enc_trunk(img, w, sc, 8)
e1.record()
torch.cuda.synchronize()
print(f"fused trunk, {n_time} images: {e0.elapsed_time(e1) / reps:.3f} ms (mean of {reps} launches)")
