"""Small decode used under compute-sanitizer (all three peaks kernels + exact select + tail)."""
import sys, torch
sys.path.insert(0, ".")
from structuredetector_b200 import ops
from structuredetector_b200.synth import DecodeConfig, make_raw, split_outputs
for (h, w, k) in ((40, 132, 30), (37, 53, 20), (24, 1028, 40)):
    cfg = DecodeConfig("san", 2, 2, 1, h, w, k, k, cfg_id=7)
    for mode in ("noise", "ties"):
        raw = make_raw(cfg, mode).cuda()
        outs = split_outputs(raw, 2, 1)
        for kw in ({}, {"warp_kernel": True}, {"exact_select": True}, {"radius": 1}):
            pk = ops.decode_packed(outs, k, k, 0.4, 0.1, **kw)
        torch.cuda.synchronize()
print("ok", int(pk.counts.sum()))
