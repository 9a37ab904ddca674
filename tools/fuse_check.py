"""Fused expand->reduce kernel (bottleneck_fuse.cu) against the unfused launches: bit-identical descriptors, and the
whole-network time at batch 256 with and without the fusion (CUDA events)."""
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from dcr_b200 import nets, synthetic, similarity   # noqa: E402
from oracle import models as om                     # noqa: E402

torch.cuda.set_device(0)
sd = om.make_sscd_state_dict(0)
batch = int(sys.argv[1]) if len(sys.argv) > 1 else 256


def run(fused: bool, img, reps: int):
    """fused: False = separate launches, True = conv3+conv1 pairs + expand-only (K = 256)"""
    os.environ["DCR_B200_TUNING"] = "1"
    os.environ.pop("DCR_NO_BLOCK_FUSION", None)
    if not fused:
        os.environ["DCR_NO_BLOCK_FUSION"] = "1"
    net = nets.build_sscd_resnet50(sd, max_batch=img.shape[0], precision="fast")
    l0 = similarity.kernel_launch_count()
    out = net(img).clone()
    launches = similarity.kernel_launch_count() - l0
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        net(img)
    e0.record()
    for _ in range(reps):
        net(img)
    e1.record()
    torch.cuda.synchronize()
    return out, e0.elapsed_time(e1) / reps, launches


small = synthetic.images(5, seed=3).cuda()
a, _, la = run(False, small, 1)
print("unfused small ok, launches", la, flush=True)
b, _, lb = run(True, small, 1)
print("fused small ok, launches", lb, "bit-identical:", bool(torch.equal(a, b)), "max diff", float((a - b).abs().max()), flush=True)
big = synthetic.images(batch, seed=4).cuda()
a, ta, _ = run(False, big, 10)
b, tb, _ = run(True, big, 10)
print(f"batch {batch}: unfused {ta:.3f} ms ({batch / ta * 1e3:.0f} img/s)  fused {tb:.3f} ms ({batch / tb * 1e3:.0f} img/s)  "
      f"bit-identical: {bool(torch.equal(a, b))}", flush=True)
