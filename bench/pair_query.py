import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from relora_b200.ops import fused as F
x = torch.randn(1024, 256, device="cuda").bfloat16(); w = torch.randn(512, 256, device="cuda").bfloat16()
o = torch.empty(1024, 512, device="cuda", dtype=torch.bfloat16)
F.gemm(x, w, o, block_n=256, pair=1); torch.cuda.synchronize()
print("pair clusters:", F._C().gemm_pair_clusters(), "SMs:", torch.cuda.get_device_properties(0).multi_processor_count)
