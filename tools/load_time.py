import os, sys, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch, amodal_depth_anything_b200 as pkg
for enc in ("vitl","vitg"):
    m = pkg.AmodalDAv2(guide_type="mask+observation", encoder=enc, pretrained=False).cuda().eval()
    torch.cuda.synchronize(); t=time.time()
    m._ensure_handle(torch.device("cuda",0)); torch.cuda.synchronize()
    print(enc, "handle build (set_weight x N + finalize) %.3f s" % (time.time()-t))
    del m
