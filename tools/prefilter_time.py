#!/usr/bin/env python
"""Time of the large-N prefilter path into the one-CTA proposal kernel: tfrpn_nms over B x K boxes with pre_nms_topn
(default 64 x 100 000, top 6000, 300 kept at IoU 0.7), CUDA events around 50 calls after 5 warm-up calls."""
import ctypes as C, os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tf-rpn_b200"))
os.environ.setdefault("TFRPN_PROP_CLUSTER", "0")
import numpy as np, torch
from tfrpn import _lib, synthetic
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
K = int(sys.argv[2]) if len(sys.argv) > 2 else 100000
dev = torch.device("cuda:0")
lib = _lib.load(); h = _lib.handle(0)
boxes, scores = synthetic.nms_boxes(np.random.default_rng(K), B, K)
b_t, s_t = torch.from_numpy(boxes).to(dev), torch.from_numpy(scores).to(dev)
nc = _lib.NmsCfg(300, 300, 0.7, float("-inf"), 0, 1, 6000)
ob = torch.empty((B, 300, 4), device=dev); os_ = torch.empty((B, 300), device=dev); oc = torch.empty((B, 300), device=dev)
ov = torch.empty((B,), dtype=torch.int32, device=dev); ok = torch.empty((B, 300), dtype=torch.int32, device=dev)
st = torch.cuda.current_stream(dev).cuda_stream
call = lambda: _lib.check(lib.tfrpn_nms(h, b_t.data_ptr(), s_t.data_ptr(), B, K, C.byref(nc), ob.data_ptr(), os_.data_ptr(),
                                        oc.data_ptr(), ov.data_ptr(), ok.data_ptr(), st))
for _ in range(5):
    call()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(50):
    call()
e1.record()
torch.cuda.synchronize()
print("prefilter nms B=%d K=%d pre_nms_topn=6000: %.1f us per call, mean valid %.1f"
      % (B, K, 1e3 * e0.elapsed_time(e1) / 50, float(ov.float().mean())))
